"""GPU tests of the guide buffers (rayz_cuda_render_guides): first-hit albedo + coverage and normal + hit distance of the camera
samples a render traces.

Small frames (160 x 90): a render with variant="bvh" runs the unstaged BVH kernel, which walks the same tree with the same
search as the guide kernel, so a render's camera segments and the guides' first hits are the same (t, sphere) per sample."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import rayz_b200
from rayz_b200 import Backend
from rayz_b200 import _abi as abi

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
W, SEED = 160, 3


def cam_for(w, defocus=0.6):
    h = int(w / rayz_b200.ASPECT_RATIO)
    return rayz_b200.Camera.init(20.0, 10.0, defocus, (13, 2, 3), (0, 0, 0), (0, 1, 0), h, w).rz, h


@pytest.fixture(scope="module")
def scene():
    return rayz_b200.random_bouncing(W, seed=42).pool.arrays()


@pytest.fixture(scope="module")
def static_scene(scene):
    """The same spheres, none of them moving: K0 (rayz_cuda_primary_ids) traces at shutter time 0 only."""
    s = dict(scene)
    s["sphere_velocity"] = np.zeros_like(scene["sphere_velocity"])
    return s


@pytest.fixture(scope="module")
def be(scene):
    b = Backend((0,))
    b.upload_scene(scene)
    yield b
    b.close()


@pytest.fixture(scope="module")
def sbe(static_scene):
    b = Backend((0,))
    b.upload_scene(static_scene)
    yield b
    b.close()


def params(h, spp, **kw):
    kw.setdefault("seed", SEED)
    kw.setdefault("variant", "bvh")
    return Backend.params(W, h, spp, kw.pop("max_depth", 50), **kw)


def _code(fn):
    with pytest.raises(abi.BackendError) as e:
        fn()
    return e.value.code


# ------------------------------------------------------------------------------- pinhole geometry in f64 (tests 2, 3, 5)
def centre_rays(cam, i, j):
    """Origin and unit direction of the ray through image point (i, j) of a pinhole camera (rz_camera_ray without jitter)."""
    o = np.array(cam.look_from[:])
    d = (np.array(cam.px_origin[:]) + np.multiply.outer(i, np.array(cam.px_du[:])) + np.multiply.outer(j, np.array(cam.px_dv[:])) - o)
    return o, d / np.linalg.norm(d, axis=-1, keepdims=True)


def sphere_hit(o, d, c, r):
    """Near root of the unit rays o + t d against spheres (c, r): (t, unit normal facing the ray); NaN where a ray misses."""
    oc = c - o
    b = np.einsum("...k,...k->...", d, oc)
    disc = b * b - (np.einsum("...k,...k->...", oc, oc) - r * r)
    t = b - np.sqrt(np.where(disc >= 0, disc, np.nan))
    n = (o + d * t[..., None] - c) / r[..., None]
    n = np.where((np.einsum("...k,...k->...", n, d) > 0)[..., None], -n, n)
    return t, n


def interior(ids):
    """Pixels whose 3 x 3 neighbourhood of K0 ids is one sphere (the image border excluded)."""
    h, w = ids.shape
    m = np.zeros_like(ids, dtype=bool)
    c = ids[1:-1, 1:-1]
    ok = c >= 0
    for dj in (-1, 0, 1):
        for di in (-1, 0, 1):
            ok &= ids[1 + dj:h - 1 + dj, 1 + di:w - 1 + di] == c
    m[1:-1, 1:-1] = ok
    return m


def solid_colour(sc, k):
    """The albedo rz_scatter gives sphere k's material wherever it is hit, or None for a checker texture."""
    mat = sc["sphere_material"][k]
    if sc["mat_kind"][mat] == abi.MAT_DIELECTRIC:
        return np.ones(3, dtype=np.float32)
    tex = sc["mat_texture"][mat]
    return sc["tex_color"][tex].astype(np.float32) if sc["tex_kind"][tex] == abi.TEX_SOLID else None


@pytest.fixture(scope="module")
def pinhole(sbe, static_scene):
    """Static scene, pinhole camera: K0's ids, the interior pixels of solid-coloured spheres, and their expected albedo."""
    cam, h = cam_for(W, defocus=0.0)
    ids = sbe.primary_ids(cam, W, h)
    inner = interior(ids)
    want = np.zeros((h, W, 3), dtype=np.float32)
    for j, i in zip(*np.nonzero(inner)):
        col = solid_colour(static_scene, ids[j, i])
        if col is None:
            inner[j, i] = False
        else:
            want[j, i] = col
    assert inner.sum() > 500, inner.sum()
    return cam, h, ids, inner, want


# ------------------------------------------------------------------------------- 1. coverage against the image
def test_coverage_is_exactly_where_the_one_sample_image_is_black(be):
    cam, h = cam_for(W)
    p = params(h, 1, max_depth=1)
    lin, _, _ = be.render(cam, p)
    alb, nrm = be.guides(cam, p)
    black = (lin[..., :3] == 0).all(axis=-1)
    assert np.array_equal(alb[..., 3] == 1, black) and np.array_equal(alb[..., 3] == 0, ~black)
    assert 0 < black.sum() < black.size
    # a missed pixel's albedo is the sky its path added, within the accumulators' 2^-32 fixed point
    assert np.abs(alb[~black][:, :3] - lin[~black][:, :3]).max() <= 2.0 ** -32
    assert (nrm[~black] == 0).all() and (nrm[black][:, 3] > 0).all()


# ------------------------------------------------------------------------------- 2. albedo exactness
def test_albedo_of_solid_sphere_interiors_is_exact(sbe, pinhole):
    cam, h, ids, inner, want = pinhole
    alb, _ = sbe.guides(cam, params(h, 8))
    m = inner & (alb[..., 3] == 1)
    assert m.sum() >= 0.99 * inner.sum()
    assert np.array_equal(alb[m][:, :3].view(np.uint32), want[m].view(np.uint32))


# ------------------------------------------------------------------------------- 3. normal and depth against f64 geometry
def test_normal_and_depth_against_f64_geometry(sbe, pinhole, static_scene):
    """One jittered sample per pixel, on the interior pixels of test 2.

    Bound: the sample's ray passes through a point of the pixel's footprint [i - 1/2, i + 1/2] x [j - 1/2, j + 1/2], and for
    an interior pixel the whole footprint lies on the same sphere (its 3 x 3 neighbours' centres do, and a sphere's image is
    convex).  Over the footprint, the angle between the normal and the centre ray's normal and the gap in hit distance are
    largest on its boundary: the normal and the distance are monotone along every line through the centre on the visible
    side of a sphere.  So the gaps are bounded by their largest values over the boundary, sampled at the four corners and the
    four edge midpoints in f64 and widened by 2 % for the curvature between those points, plus the FP32 error of the search
    (sphere test and camera ray: a few ulp of t ~ 13, 2e-5 here) and of the f32 normal (1e-6 rad)."""
    cam, h, ids, inner, _ = pinhole
    _, nrm = sbe.guides(cam, params(h, 1))
    j, i = np.nonzero(inner)
    k = ids[j, i]
    c = static_scene["sphere_center"][k]
    r = static_scene["sphere_radius"][k]
    o, d = centre_rays(cam, i.astype(np.float64), j.astype(np.float64))
    t0, n0 = sphere_hit(o, d, c, r)
    assert np.isfinite(t0).all()
    ang_max = np.zeros_like(t0)
    dt_max = np.zeros_like(t0)
    for di, dj in ((-.5, -.5), (.5, -.5), (-.5, .5), (.5, .5), (0, -.5), (0, .5), (-.5, 0), (.5, 0)):
        _, dd = centre_rays(cam, i + di, j + dj)
        t1, n1 = sphere_hit(o, dd, c, r)
        assert np.isfinite(t1).all()
        ang_max = np.maximum(ang_max, np.arccos(np.clip(np.einsum("pk,pk->p", n0, n1), -1, 1)))
        dt_max = np.maximum(dt_max, np.abs(t1 - t0))
    got = nrm[j, i].astype(np.float64)
    assert np.abs(np.linalg.norm(got[:, :3], axis=-1) - 1).max() < 1e-6
    ang = np.arccos(np.clip(np.einsum("pk,pk->p", got[:, :3] / np.linalg.norm(got[:, :3], axis=-1, keepdims=True), n0), -1, 1))
    assert (ang <= ang_max * 1.02 + 1e-6).all(), float((ang - ang_max).max())
    assert (np.abs(got[:, 3] - t0) <= dt_max * 1.02 + 2e-5).all(), float((np.abs(got[:, 3] - t0) - dt_max).max())
    assert ang.max() > 0 and ang_max.max() < 0.5   # the bound is not vacuous


# ------------------------------------------------------------------------------- 4. invariance
@pytest.mark.parametrize("count,band", [(3, 1), (3, 4), (8, 1), (8, 4)])
def test_shards_assemble_the_full_frame(be, count, band):
    cam, h = cam_for(W)
    full = be.guides(cam, params(h, 4))
    parts = [np.full_like(x, np.nan) for x in full]
    for s in range(count):
        got = be.guides(cam, params(h, 4, shard_index=s, shard_count=count, band_rows=band))
        rows = [j for j in range(h) if (j // band) % count == s]
        assert got[0].shape[0] == len(rows)
        for f, x in zip(parts, got):
            f[rows] = x
    for f, x in zip(parts, full):
        assert np.array_equal(f.view(np.uint32), x.view(np.uint32))


def test_two_calls_are_identical_and_the_variant_does_not_matter(be):
    cam, h = cam_for(W)
    a = be.guides(cam, params(h, 5))
    for v in ("bvh", "auto", "mega", "mega_single", "wavefront"):
        b = be.guides(cam, params(h, 5, variant=v, max_depth=1 if v == "bvh" else 7, collect_stats=v == "auto"))
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
        want = be.guides(cam, params(h, 4, **kw))
        got = many.guides(cam, params(h, 4, **kw))
        for x, y in zip(got, want):
            assert np.array_equal(x.view(np.uint32), y.view(np.uint32)), kw
    many.close()


# ------------------------------------------------------------------------------- 5. sample ranges
def test_a_sample_range_is_the_mean_of_its_samples(be):
    cam, h = cam_for(W)
    o = 6
    alb, nrm = be.guides(cam, params(h, 4, sample_offset=o))
    one = [be.guides(cam, params(h, 1, sample_offset=o + s)) for s in range(4)]
    a = [x[0].astype(np.float64) for x in one]
    n = [x[1].astype(np.float64) for x in one]
    hit = [x[..., 3] for x in a]   # 0 or 1 per sample
    sum_a = ((a[0] + a[1]) + a[2]) + a[3]   # the kernel's order
    sum_n = ((n[0][..., :3] + n[1][..., :3]) + n[2][..., :3]) + n[3][..., :3]
    sum_t = ((n[0][..., 3] * hit[0] + n[1][..., 3] * hit[1]) + n[2][..., 3] * hit[2]) + n[3][..., 3] * hit[3]
    cnt = hit[0] + hit[1] + hit[2] + hit[3]
    want_a = (sum_a / 4).astype(np.float32)
    want_n = np.concatenate([sum_n / 4, np.where(cnt > 0, sum_t / np.maximum(cnt, 1), 0)[..., None]], axis=-1).astype(np.float32)
    for got, want in ((alb, want_a), (nrm, want_n)):
        ulp = np.spacing(np.abs(want))
        assert (np.abs(got - want) <= ulp).all()
    assert ((cnt > 0) & (cnt < 4)).any()   # some pixels are edges: the range is a real mean


def test_another_seed_changes_edges_not_solid_interiors(sbe, pinhole):
    cam, h, ids, inner, want = pinhole
    a1, n1 = sbe.guides(cam, params(h, 4, seed=1))
    a2, n2 = sbe.guides(cam, params(h, 4, seed=2))
    assert not np.array_equal(a1, a2) and not np.array_equal(n1, n2)
    assert np.array_equal(a1[inner], a2[inner])


# ------------------------------------------------------------------------------- 6. no side effects
def test_guides_leave_the_accumulated_frame_alone(be):
    cam, h = cam_for(W)

    def sequence(with_guides):
        be.render(cam, params(h, 4, moments=True))
        if with_guides:
            be.guides(cam, params(h, 7, seed=SEED + 1, sample_offset=2))
        lin, rgb8, _ = be.render(cam, params(h, 4, sample_offset=4, moments=True, accumulate=True))
        err, nz = be.noise(0.01)
        return lin, rgb8, err, nz, be.pixel_samples()

    want, got = sequence(False), sequence(True)
    for x, y in zip(got, want):
        assert np.array_equal(x, y) if isinstance(x, np.ndarray) else x == y


def test_guides_leave_an_adaptive_frame_alone(be):
    cam, h = cam_for(W)
    be.render(cam, params(h, 4, moments=True))
    target = float(np.quantile(be.noise(0.0)[0], 0.5) / 4)   # the sky meets it at once, the noisiest pixels never
    be.render_to_noise(cam, params(h, 4), target, 64, adaptive=True)
    counts, (err, nz) = be.pixel_samples(), be.noise(target)
    assert len(np.unique(counts)) > 1
    be.guides(cam, params(h, 4))
    err2, nz2 = be.noise(target)
    assert np.array_equal(be.pixel_samples(), counts) and np.array_equal(err2, err) and nz2 == nz


def test_guides_leave_stats_and_timing_alone(be):
    cam, h = cam_for(W)
    be.render(cam, params(h, 4, collect_stats=True))
    s, t = be.stats(), be.timing()
    be.guides(cam, params(h, 4, collect_stats=True))
    assert be.stats() == s and be.timing() == t


# ------------------------------------------------------------------------------- 7. refusals and faults
def test_refusals(be, scene):
    cam, h = cam_for(W)
    lib = be.lib
    out = np.zeros((h, W, 4), dtype=np.float32)

    def call(b, p, c=cam):
        return b.lib.rayz_cuda_render_guides(b._h, C.byref(c) if c is not None else None, C.byref(p) if p is not None else None,
                                             out.ctypes.data, out.ctypes.data)

    def refused(code, rc, text):
        assert rc == code, (rc, lib.rayz_cuda_last_error())
        msg = lib.rayz_cuda_last_error()
        assert msg.startswith(b"guides:") and text in msg, msg

    refused(-1, call(be, None), b"NULL")
    refused(-1, call(be, params(h, 4), None), b"NULL")
    fresh = Backend((0,))
    refused(-6, call(fresh, params(h, 4)), b"rayz_cuda_upload_scene")
    fresh.close()
    refused(-1, call(be, params(h, 0)), b"spp")
    big = params(h, 1)
    big.width, big.height = 65536, 32768
    refused(-1, call(be, big), b"image too large")
    bad = params(h, 1)
    bad.variant = 9
    refused(-1, call(be, bad), b"unknown variant")
    refused(-1, call(be, params(h, 1, shard_index=3, shard_count=3)), b"shard_index")
    refused(-1, call(be, params(h, 1, accumulate=True)), b"RZ_RENDER_ACCUMULATE")
    ad = params(h, 1)
    ad.flags |= abi.RENDER_ADAPTIVE
    refused(-1, call(be, ad), b"RZ_RENDER_ADAPTIVE")
    assert (out == 0).all()

    # a traversal stack the kernel believes holds one entry overflows: RZ_ERR_INTERNAL, and the context stays usable
    be.set_tuning(debug_stack_cap=1)
    try:
        refused(-7, call(be, params(h, 2)), b"traversal-stack overflow")
    finally:
        be.set_tuning(debug_stack_cap=0)
    a, _ = be.guides(cam, params(h, 2))
    assert np.isfinite(a).all()
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


def test_cpp_host_guides_match_backend(tmp_path):
    subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "host")], check=True)
    exe = os.path.join(ROOT, "host", "_build", "rayz_host")
    prefix = str(tmp_path / "g")
    r = subprocess.run([exe, str(W), str(tmp_path / "o.ppm"), "--spp", "4", "--seed", "42", "--render-seed", "5", "--guides", prefix],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    t = rayz_b200.random_bouncing(W, seed=42)
    t.samples_per_px, t.seed = 4, 5
    alb, nrm = t.render_guides()
    assert t.albedo is alb and t.normal is nrm
    assert np.array_equal(read_pfm(prefix + "_albedo.pfm"), alb[..., :3])
    assert np.array_equal(read_pfm(prefix + "_normal.pfm"), nrm[..., :3])
    assert np.array_equal(read_pfm(prefix + "_depth.pfm")[..., 0], nrm[..., 3])
    t.backend.close()
