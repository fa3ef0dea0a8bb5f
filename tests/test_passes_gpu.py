"""GPU tests of light-path passes (RZ_RENDER_PASSES, include/rayz_cuda.h "Light-path passes").

1. The flag changes no image: linear, rgb8 and the noise estimate are bit-identical with and without it, for every variant and
   sampler; the passes sum to the linear frame to f32 rounding; the brute-force family gives bit-identical passes, so does
   the BVH family, and at >= 2^26 paths the staged pipelines' passes equal the unstaged kernels'.
2. One path per pixel: at most one nonzero pass, bit-identical to the pixel's linear value.
3. The right pass: every robust replayed path lands in rz_pass_of(hits, first hit's kind), with zero exceptions.
4. Batches, shards and devices reproduce the passes bit for bit; a batch that drops or adds the bit is refused.
5. Adaptive frames (plain and pooled): a pixel with count c has the passes of a uniform c-spp render.
6. Refusals, with nothing touched.
7. The C++ host writes the seven passes as PFM files."""
import os
import subprocess

import numpy as np
import pytest

import oracle
import rayz_b200
from passes_replay import pass_of, replay_first
from rayz_b200 import Backend
from rayz_b200 import _abi as abi
from replay_scenes import all_materials, config1

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SEED = 11
SAMPLERS = {"philox": {}, "sobol": {"sobol": True}, "sobol-rqmc": {"sobol": True, "rqmc": True, "moments": True}}
VARIANTS = [("auto", {}), ("mega", {"tail_brute": 0}), ("mega", {"tail_brute": 1}), ("mega_single", {}), ("wavefront", {}),
            ("bvh", {})]
BRUTE = [("mega", {"tail_brute": 1}), ("mega_single", {}), ("wavefront", {})]
DEFAULT_TUNING = {"tail_brute": 0, "bvh_staged": 1}


@pytest.fixture(scope="module")
def be():
    b = Backend((0,))
    yield b
    b.set_tuning(**DEFAULT_TUNING)
    b.close()


@pytest.fixture(scope="module")
def small():
    arrays, cam = config1(160, 90)
    return arrays, cam, 160, 90


def params(w, h, spp, sampler="philox", **kw):
    kw.setdefault("seed", SEED)
    kw.setdefault("variant", "bvh")
    kw.setdefault("moments", True)
    s = dict(SAMPLERS[sampler])
    kw["moments"] = s.pop("moments", False) or kw["moments"]
    return Backend.params(w, h, spp, kw.pop("max_depth", 50), **kw, **s)


def check_sum(P, lin, label):
    """The seven passes sum to the linear frame to f32 rounding (at most 8 ulp per channel), and a = 1 everywhere."""
    s = P[..., :3].astype(np.float64).sum(axis=0)
    ref = lin[..., :3].astype(np.float64)
    ulp = np.spacing(np.abs(lin[..., :3])).astype(np.float64)
    bad = np.abs(s - ref) > 8 * ulp
    assert not bad.any(), f"{label}: {int(bad.sum())} channels off by more than 8 ulp, worst {np.max(np.abs(s - ref) / np.maximum(ulp, 1e-45))} ulp"
    assert (P[..., 3] == 1.0).all()


# ------------------------------------------------------------------------------- 1. no image changes; sums; families
@pytest.mark.parametrize("sampler", list(SAMPLERS))
def test_flag_changes_no_image_and_passes_sum_to_it(be, small, sampler):
    arrays, cam, w, h = small
    be.upload_scene(arrays)
    got = {}
    try:
        for variant, tun in VARIANTS:
            be.set_tuning(**{**DEFAULT_TUNING, **tun})
            lin0, rgb0, _ = be.render(cam, params(w, h, 8, sampler, variant=variant))
            err0, nz0 = be.noise(0.01)
            lin1, rgb1, _ = be.render(cam, params(w, h, 8, sampler, variant=variant, passes=True))
            err1, nz1 = be.noise(0.01)
            label = f"{sampler} {variant} {tun}"
            assert np.array_equal(lin0.view(np.uint32), lin1.view(np.uint32)), label
            assert np.array_equal(rgb0, rgb1) and np.array_equal(err0.view(np.uint32), err1.view(np.uint32)) and nz0 == nz1, label
            P = be.passes()
            assert P.shape == (7, h, w, 4)
            check_sum(P, lin1, label)
            assert (P[..., :3] > 0).any(axis=(1, 2, 3)).sum() >= 4, label
            got[(variant, tuple(tun.items()))] = P
    finally:
        be.set_tuning(**DEFAULT_TUNING)
    key = lambda v, t: (v, tuple(t.items()))
    ref = got[key(*BRUTE[0])]
    for v, t in BRUTE[1:]:
        assert np.array_equal(got[key(v, t)], ref), (sampler, v, t)
    assert np.array_equal(got[key("auto", {})], got[key("bvh", {})]), sampler   # AUTO runs the BVH kernel at this size


@pytest.mark.parametrize("sampler", ["philox", "sobol-rqmc"])
def test_staged_pipelines_at_flagship_size(be, sampler):
    """Frames of >= 2^26 paths run the staged forms: AUTO's primary kernel -> sorted stages -> BVH tail, and K3's camera stage +
    queue.  The image does not change with the flag, the passes sum to it, and the staged K3's passes equal the unstaged K3's."""
    t = rayz_b200.random_bouncing(1200, seed=42)
    be.upload_scene(t.pool.arrays())
    cam, w, h, spp = t.camera.rz, 1200, 675, 84   # 68 M paths
    try:
        lin0, rgb0, _ = be.render(cam, params(w, h, spp, sampler, variant="auto"))
        lin1, rgb1, _ = be.render(cam, params(w, h, spp, sampler, variant="auto", passes=True))
        assert be.timing()["passes"] > 0   # the staged form ran
        assert np.array_equal(lin0.view(np.uint32), lin1.view(np.uint32)) and np.array_equal(rgb0, rgb1)
        check_sum(be.passes(), lin1, f"auto staged {sampler}")
        staged = {}
        for st in (1, 0):
            be.set_tuning(bvh_staged=st)
            lin, _, _ = be.render(cam, params(w, h, spp, sampler, variant="bvh", passes=True))
            staged[st] = (lin, be.passes())
        assert np.array_equal(staged[0][0], staged[1][0]) and np.array_equal(staged[0][1], staged[1][1])
        check_sum(staged[1][1], staged[1][0], f"bvh staged {sampler}")
    finally:
        be.set_tuning(**DEFAULT_TUNING)


# ------------------------------------------------------------------------------- 2 + 3. one path per pass, the right pass
def _scenes():
    a1, c1 = config1(160, 90)
    ag, cg = config1(160, 90, glass_heavy=True)
    am, cams, wm, hm = all_materials()
    return {"config1": (a1, c1, 160, 90), "glass": (ag, cg, 160, 90), "all_outside": (am, cams["outside"], wm, hm),
            "all_in_glass": (am, cams["in_glass"], wm, hm)}


SCENES = _scenes()


@pytest.mark.parametrize("name", list(SCENES))
@pytest.mark.parametrize("sampler", list(SAMPLERS))
def test_each_path_lands_in_its_pass(be, name, sampler):
    arrays, cam, w, h = SCENES[name]
    spp = 2 if sampler == "sobol-rqmc" else 1
    sc = oracle.Scene.from_arrays(arrays)
    rep = sc.replay(cam, w, h, 0, spp, 50, seed=SEED, sampler=sampler)
    first, _ = replay_first(sc, cam, w, h, 0, spp, seed=SEED, sampler=sampler)
    hits = rep["hits"].sum(axis=-1)
    sky = rep["end"] == oracle.END_SKY
    lit = sky & (rep["rgb"].max(axis=-1) > 1e-6)                   # adds a nonzero fixed-point value
    dark = ~sky | (rep["rgb"].max(axis=-1) == 0)                   # adds nothing
    want = np.zeros((h, w, 7), bool)                              # the passes the pixel's paths add to
    pidx = pass_of(hits, first)
    yy, xx = np.indices((h, w))
    for s in range(spp):
        want[yy, xx, pidx[..., s]] |= lit[..., s]
    judged = (rep["robust"] & (lit | dark)).all(axis=-1)           # every path of the pixel robust and unambiguous
    be.upload_scene(arrays)
    checked = 0
    try:
        for variant, tun in VARIANTS:
            be.set_tuning(**{**DEFAULT_TUNING, **tun})
            lin, _, _ = be.render(cam, params(w, h, spp, sampler, variant=variant, passes=True))
            P = be.passes()
            nonzero = (P[..., :3] != 0).any(axis=-1).transpose(1, 2, 0)   # [h, w, 7]
            label = f"{name} {sampler} {variant} {tun}"
            if spp == 1:   # one path per pixel: at most one pass, and it is the pixel's value bit for bit
                assert (nonzero.sum(axis=-1) <= 1).all(), label
                one = nonzero.any(axis=-1)
                k = nonzero.argmax(axis=-1)
                sel = np.take_along_axis(P.transpose(1, 2, 0, 3), k[..., None, None], axis=2)[:, :, 0, :3]
                assert np.array_equal(sel[one].view(np.uint32), lin[..., :3][one].view(np.uint32)), label
                assert not nonzero[(lin[..., :3] == 0).all(axis=-1)].any(), label
            check_sum(P, lin, label)
            bad = judged & (nonzero != want).any(axis=-1)
            assert not bad.any(), f"{label}: {int(bad.sum())} robust pixels in the wrong pass, first at {np.argwhere(bad)[0]}"
            checked += int(judged.sum())
    finally:
        be.set_tuning(**DEFAULT_TUNING)
    print(f"  {name} {sampler}: {checked} robust pixel-checks, fragile {1 - rep['robust'].mean():.2%}")
    assert judged.mean() > 0.9


# ------------------------------------------------------------------------------- 4. batches, shards, devices
@pytest.mark.parametrize("variant", ["bvh", "mega_single"])
@pytest.mark.parametrize("sampler", ["philox", "sobol-rqmc"])
def test_batches_reproduce_one_render_and_refuse_a_changed_bit(be, small, variant, sampler):
    arrays, cam, w, h = small
    be.upload_scene(arrays)
    be.render(cam, params(w, h, 12, sampler, variant=variant, passes=True))
    whole = be.passes()
    be.render(cam, params(w, h, 4, sampler, variant=variant, passes=True))
    be.render(cam, params(w, h, 8, sampler, variant=variant, passes=True, sample_offset=4, accumulate=True))
    assert np.array_equal(be.passes(), whole)
    for flip in ("drop", "add"):
        base = params(w, h, 4, sampler, variant=variant, passes=flip == "drop")
        be.render(cam, base)
        before_err = be.noise()[0]
        before = be.passes() if flip == "drop" else None
        nxt = params(w, h, 8, sampler, variant=variant, passes=flip == "add", sample_offset=4, accumulate=True)
        with pytest.raises(abi.BackendError) as e:
            be.render(cam, nxt)
        assert e.value.code == -1 and "RZ_RENDER_PASSES bit differs" in str(e.value), str(e.value)
        assert np.array_equal(be.noise()[0], before_err)   # the sums are untouched
        if before is not None:
            assert np.array_equal(be.passes(), before)


def _global_rows(h, s, count, band):
    rows = np.arange(h)
    return rows[(rows // band) % count == s]


def test_shards_assemble_the_full_frame(be, small):
    arrays, cam, w, h = small
    be.upload_scene(arrays)
    band, count = 3, 3
    be.render(cam, params(w, h, 6, variant="bvh", passes=True, band_rows=band))
    full = be.passes()
    for s in range(count):
        be.render(cam, params(w, h, 6, variant="bvh", passes=True, band_rows=band, shard_index=s, shard_count=count))
        assert np.array_equal(be.passes(), full[:, _global_rows(h, s, count, band)]), s


def _n_gpus():
    import torch
    return torch.cuda.device_count()


@pytest.mark.skipif("_n_gpus() < 2")
def test_two_devices_equal_one(be, small):
    arrays, cam, w, h = small
    be.upload_scene(arrays)
    be.render(cam, params(w, h, 6, variant="bvh", passes=True))
    one = be.passes()
    many = Backend((0, 1))
    try:
        many.upload_scene(arrays)
        many.render(cam, params(w, h, 6, variant="bvh", passes=True))
        assert np.array_equal(many.passes(), one)
    finally:
        many.close()


# ------------------------------------------------------------------------------- 5. adaptive
@pytest.mark.parametrize("pooled", [False, True])
def test_adaptive_pixels_equal_uniform_renders_of_their_count(be, small, pooled):
    arrays, cam, w, h = small
    be.upload_scene(arrays)
    be.render(cam, params(w, h, 4, variant="bvh"))
    target = float(np.quantile(be.noise()[0], 0.5) / 3)
    lin, _, _, _ = be.render_to_noise(cam, params(w, h, 4, variant="bvh", passes=True), target, 64, adaptive=True, pooled=pooled)
    P = be.passes()
    counts = be.pixel_samples()
    check_sum(P, lin, f"adaptive pooled={pooled}")
    distinct = np.unique(counts)
    assert len(distinct) >= 3, distinct
    for c in distinct:
        m = counts == c
        be.render(cam, params(w, h, int(c), variant="bvh", passes=True))
        assert np.array_equal(P[:, m], be.passes()[:, m]), (pooled, c)


# ------------------------------------------------------------------------------- 6. refusals
def test_refusals_touch_nothing(be, small):
    arrays, cam, w, h = small
    be.upload_scene(arrays)
    be.render(cam, params(w, h, 4))
    with pytest.raises(abi.BackendError) as e:
        be.passes()
    assert e.value.code == -1 and "without RZ_RENDER_PASSES" in str(e.value)
    be.render(cam, params(w, h, 4, passes=True))
    P, err = be.passes(), be.noise()[0]

    def refused(call, text):
        with pytest.raises(abi.BackendError) as e:
            call()
        assert e.value.code == -1 and text in str(e.value), str(e.value)
        assert np.array_equal(be.passes(), P) and np.array_equal(be.noise()[0], err)

    refused(lambda: be.guides(cam, params(w, h, 4, passes=True)), "guides: RZ_RENDER_PASSES")
    deep = params(w, h, 4, passes=True, max_depth=1 << 29)
    refused(lambda: be.render(cam, deep), "RZ_RENDER_PASSES requires max_depth <= 2^29 - 1")
    refused(lambda: be.render_to_noise(cam, deep, 0.01, 8), "RZ_RENDER_PASSES requires max_depth")
    refused(lambda: be.reserve(deep), "RZ_RENDER_PASSES requires max_depth")
    be.render(cam, params(w, h, 4, passes=True, max_depth=(1 << 29) - 1))   # the largest accepted depth renders


# ------------------------------------------------------------------------------- 7. the C++ host
def read_pfm(path):
    raw = open(path, "rb").read()
    tag, dims, scale, body = raw.split(b"\n", 3)
    w, h = (int(x) for x in dims.split())
    assert tag == b"PF" and float(scale) == -1.0
    return np.frombuffer(body, dtype="<f4").reshape(h, w, 3)[::-1]


def test_cpp_host_writes_the_passes(tmp_path):
    subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "host")], check=True)
    exe = os.path.join(ROOT, "host", "_build", "rayz_host")
    prefix, W = str(tmp_path / "p"), 200
    r = subprocess.run([exe, str(W), str(tmp_path / "o.ppm"), "--spp", "4", "--seed", "42", "--render-seed", "5", "--passes", prefix,
                        "--dump-linear", str(tmp_path / "lin.f32")], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    H = int(W / rayz_b200.ASPECT_RATIO)
    lin = np.fromfile(tmp_path / "lin.f32", dtype=np.float32).reshape(H, W, 4)
    planes = np.stack([read_pfm(f"{prefix}_{n}.pfm") for n in abi.PASS_NAMES])
    P = np.concatenate([planes, np.ones(planes.shape[:3] + (1,), np.float32)], axis=-1)
    check_sum(P, lin, "rayz_host --passes")
    assert (planes > 0).any(axis=(1, 2, 3)).sum() >= 4
