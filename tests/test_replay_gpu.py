"""GPU tests: every kernel family's paths against the oracle's f64 replay of the same paths (oracle Scene.replay).

Each uniform the kernels draw is a pure function of (seed, pixel, sample, bounce), so a 1-spp frame is one path per pixel
and the replay traces exactly those paths in f64.  A robust path (no decision within f32 rounding of a boundary, and no
change of events under perturbed replays) must agree within its own tolerance, with zero exceptions; the counters of
collect_stats must equal the replay's up to what the fragile paths can move; the per-pixel noise estimate must equal
rz_pixel_err's formula on the replay's path values.  One replay per (scene, camera, sampler, depth, t_min, frames) is
shared by every kernel variant, tuning and stats build that renders it.  The staged BVH pipeline (K3's camera stage and
queue) runs only on frames of >= 2^26 paths, far beyond what the replay traces; it is covered through
test_gpu_parity's bitwise staged == unstaged comparison."""
import functools

import math

import numpy as np
import pytest

import oracle
import rayz_b200
from rayz_b200 import Backend
from rayz_b200 import _abi as abi
from replay_scenes import all_materials, compare_paths, config1, count_stats, metal_floor, stat_slack

pytestmark = pytest.mark.gpu

# (variant, tuning): every path-kernel family and the tuning switch that picks another kernel instance at these frame sizes
# (the staged K1's tail: the BVH kernel or brute force).  bvh_staged changes nothing below 2^26 paths (see above).
VARIANTS = [("auto", {}), ("mega", {"tail_brute": 0}), ("mega", {"tail_brute": 1}), ("mega_single", {}), ("wavefront", {}),
            ("bvh", {})]
DEFAULT_TUNING = {"tail_brute": 0}
SEED = 11


@pytest.fixture(scope="module")
def be():
    b = Backend((0,))
    yield b
    b.close()


@functools.lru_cache(maxsize=None)
def _scene(name):
    if name in ("config1", "glass"):
        arrays, cam = config1(glass_heavy=name == "glass")
        return arrays, {"default": cam}, 317, 178
    if name == "metal_floor":
        arrays, cam, w, h = metal_floor()
        return arrays, {"default": cam}, w, h
    return all_materials()


@functools.lru_cache(maxsize=None)
def _replay(scene, camname, sampler, depth, t_min, offset, spp):
    arrays, cams, w, h = _scene(scene)
    return oracle.Scene.from_arrays(arrays).replay(cams[camname], w, h, offset, spp, depth, seed=SEED, t_min=t_min, sampler=sampler)


def _pixels(rep):
    """A replay of spp paths per pixel as one entry per pixel: the mean radiance, robust when every path is."""
    spp = rep["rgb"].shape[2]
    return {"rgb": rep["rgb"].mean(axis=2, keepdims=True), "tol": rep["tol"].mean(axis=2, keepdims=True),
            "robust": rep["robust"].all(axis=2, keepdims=True), "segs": rep["segs"].sum(axis=2, keepdims=True),
            "end": rep["end"][:, :, :1], "hits": rep["hits"].sum(axis=2, keepdims=True), "hash": rep["hash"][:, :, :1],
            "spp": spp}


def _check_stats(be, rep, depth, label):
    """collect_stats against the replay's counters: each may differ by at most what the fragile paths can move it.  Returns
    the counters whose slack is at most STATS_SLACK_MAX of their count (the ones this frame checks meaningfully)."""
    got, want, slack = be.stats(), count_stats(rep), stat_slack(rep, depth)
    diffs = {k: int(got[k]) - want[k] for k in want}
    print(f"  {label} stats diff {diffs}, fragile slack {slack}")
    for k in want:
        assert abs(diffs[k]) <= slack[k], f"{label}: stats {k} = {got[k]}, replay {want[k]}, fragile paths allow {slack[k]}"
    return {k for k in want if want[k] > 0 and slack[k] <= STATS_SLACK_MAX * want[k]}


def _check_paths_and_ends(be, rep, label):
    """Deep frames: a fragile path may add up to a full depth of segments, so the other counters are checked on shallow
    frames (test_stats_equal_the_replay); here the path count is exact and every path ends once."""
    got = be.stats()
    n = rep["segs"].size
    assert got["paths"] == n and got["ended_sky"] + got["ended_absorbed"] + got["ended_depth"] == n, (label, got)


def _run_case(be, scene, camname, sampler, depth, t_min, frames, variants, fragile_max):
    """frames: (sample_offset, spp) pairs.  Renders each frame with every variant, with and without collect_stats."""
    arrays, cams, w, h = _scene(scene)
    be.upload_scene(arrays)
    worst = 0.0
    try:
        for off, spp in frames:
            rep = _replay(scene, camname, sampler, depth, t_min, off, spp)
            pix = _pixels(rep)
            frag = 1.0 - float(rep["robust"].mean())
            assert frag <= fragile_max, f"fragile fraction {frag:.3%} above {fragile_max:.1%}"
            for variant, tun in variants:
                be.set_tuning(**{**DEFAULT_TUNING, **tun})
                for stats in (True, False):
                    p = Backend.params(w, h, spp, depth, seed=SEED, sample_offset=off, variant=variant, t_min=t_min,
                                       collect_stats=stats, sobol=sampler != "philox", rqmc=sampler == "sobol-rqmc",
                                       moments=sampler == "sobol-rqmc")
                    lin, _, n = be.render(cams[camname], p, want_rgb8=False)
                    assert n == w * h * spp
                    label = (f"{scene}/{camname} {sampler} depth {depth} t_min {t_min} frame ({off}, {spp}) {variant} {tun} "
                             f"stats {stats}")
                    worst = max(worst, compare_paths(pix, lin[:, :, None, :3], label))
                    if stats:
                        _check_paths_and_ends(be, rep, label)
    finally:
        be.set_tuning(**DEFAULT_TUNING)
    return worst


# Fragile fractions of these frames (measured by the replay itself, so known before any GPU run): config 1 about 3 %, the
# glass-heavy scene about 5 %, the all-materials scene 0.3-2.8 %.  Bars: about 1.5 x.
def test_config1_philox_every_kernel(be):
    _run_case(be, "config1", "default", "philox", 50, 0.0, [(0, 1), (1, 1)], VARIANTS, 0.045)


def test_config1_sobol_every_kernel(be):
    _run_case(be, "config1", "default", "sobol", 50, 0.0, [(0, 1), (5, 1)], VARIANTS, 0.045)


def test_config1_sobol_rqmc_every_kernel(be):
    """RQMC needs moments and an even spp: 2-spp frames at even offsets, both replicates in each pixel."""
    _run_case(be, "config1", "default", "sobol-rqmc", 50, 0.0, [(0, 2), (6, 2)], VARIANTS, 0.045)


@pytest.mark.parametrize("sampler", ["philox", "sobol"])
def test_glass_heavy_scene(be, sampler):
    _run_case(be, "glass", "default", sampler, 50, 0.0, [(0, 1)], VARIANTS, 0.08)


@pytest.mark.parametrize("depth", [0, 1, 2, 50])
def test_all_materials_depths(be, depth):
    _run_case(be, "allmat", "outside", "philox", depth, 0.0, [(0, 1)], VARIANTS, 0.04)


def test_all_materials_sobol_and_camera_in_glass(be):
    _run_case(be, "allmat", "outside", "sobol", 2, 0.0, [(2, 1)], VARIANTS, 0.04)
    _run_case(be, "allmat", "in_glass", "philox", 50, 1e-3, [(0, 1)], VARIANTS, 0.04)


# ------------------------------------------------------------------------------- counters
# At depth 2 a fragile path can move a counter by at most a few units, against thousands of counted events.  A counter is
# checked meaningfully in a frame when its slack is at most this fraction of its count; every counter must be, in some frame
# of every sampler (the metal floor is there for ended_absorbed, which is rare in the other scenes).
STATS_SLACK_MAX = 0.1


@pytest.mark.parametrize("sampler", ["philox", "sobol", "sobol-rqmc"])
def test_stats_equal_the_replay(be, sampler):
    """Each sampler's stats instance of every kernel family: RzStats equal to the replay's counters up to the fragile paths."""
    frame = (0, 2) if sampler == "sobol-rqmc" else (0, 1)
    covered = set()
    try:
        for scene in ("config1", "glass", "metal_floor"):
            arrays, cams, w, h = _scene(scene)
            be.upload_scene(arrays)
            rep = _replay(scene, "default", sampler, 2, 0.0, *frame)
            for variant, tun in VARIANTS:
                be.set_tuning(**{**DEFAULT_TUNING, **tun})
                p = Backend.params(w, h, frame[1], 2, seed=SEED, sample_offset=frame[0], variant=variant, collect_stats=True,
                                   sobol=sampler != "philox", rqmc=sampler == "sobol-rqmc", moments=sampler == "sobol-rqmc")
                lin, _, _ = be.render(cams["default"], p, want_rgb8=False)
                label = f"{scene} {sampler} depth 2 {variant} {tun}"
                compare_paths(_pixels(rep), lin[:, :, None, :3], label)
                covered |= _check_stats(be, rep, 2, label)
    finally:
        be.set_tuning(**DEFAULT_TUNING)
    missing = set(count_stats(rep)) - covered
    assert not missing, f"{sampler}: no frame checks {sorted(missing)} with a slack below {STATS_SLACK_MAX:.0%} of the count"


# ------------------------------------------------------------------------------- the checker lattice, exactly
# The lattice is tested in f64 on the f64 hit point with the f64 1 / scale (rz_checker2, and the record that carries 1 / scale
# as two f32 words).  Random paths cannot show an f32 1 / scale: it moves the lattice by about u |p|, no more than the f32
# error of a random hit point.  A camera ray along -y from an f32-exact origin is exact (px_du = px_dv = 0: every pixel traces
# it), so its hit point is too, and its x coordinate is chosen where floor(x / 0.3) in f64 and with an f32 1 / scale differ.
CHECKER_X = 8192.0 + 1678029 * 2.0 ** -10     # 9830.7001953125: 6.5e-4 of a cell past a boundary in f64, 1.3e-4 before it in f32


def test_checker_of_two_solids_uses_the_f64_inverse_scale(be):
    inv = 1.0 / 0.3
    assert float(np.float32(CHECKER_X)) == CHECKER_X
    assert math.floor(CHECKER_X * inv) != math.floor(CHECKER_X * float(np.float32(inv))), "the case would not tell"
    y_top, z = 0.15, 0.5
    cell = math.floor(CHECKER_X * inv) + math.floor(y_top * inv) + math.floor(z * inv)
    even = cell % 2 == 0
    pool = rayz_b200.MemPool()
    ck = pool.add_checker(0.3, pool.add_solid((0.9, 0.05, 0.05)), pool.add_solid((0.05, 0.05, 0.9)))
    pool.add_sphere((CHECKER_X, y_top - 1.0, z), 1.0, pool.add_diffuse(ck))
    cam = abi.RzCamera()
    cam.look_from[:] = (CHECKER_X, 5.0, z)
    cam.px_origin[:] = (CHECKER_X, 4.0, z)
    be.upload_scene(pool.arrays())
    w, h = 16, 8
    for variant, tun in VARIANTS:
        be.set_tuning(**{**DEFAULT_TUNING, **tun})
        try:
            lin, _, _ = be.render(cam, Backend.params(w, h, 1, 2, seed=SEED, variant=variant), want_rgb8=False)
        finally:
            be.set_tuning(**DEFAULT_TUNING)
        red = lin[..., 0] > lin[..., 2]
        assert (lin[..., :3] > 0).any(axis=-1).all(), "every path ends in the sky after one diffuse bounce"
        assert (red == even).all(), f"{variant} {tun}: {int((red != even).sum())} of {w * h} pixels in the wrong checker cell"


# ------------------------------------------------------------------------------- the noise estimate
def _err2_bound(y, tol, n):
    """rz_pixel_err's e^2 = s^2 / (4 n max(Ybar, 1e-4)) per pixel from the replay's path luminances y [.., n], and how far the
    kernels' f32 values (each path within tol of the replay's) can move it."""
    ybar = y.mean(-1)
    q3 = np.minimum(y * y, 1048576.0).mean(-1)
    s2 = np.maximum(0.0, q3 - ybar * ybar) * n / (n - 1)
    den = 4.0 * n * np.maximum(ybar, 1e-4)
    e2 = s2 / den
    dy = tol.mean(-1) + 1e-9                                   # + the 2^-32 fixed point
    dq3 = (2.0 * y * tol + tol * tol).mean(-1) + 1e-9
    ds2 = (dq3 + 2.0 * ybar * dy + dy * dy) * n / (n - 1)
    dinv = np.abs(1.0 / np.maximum(ybar - dy, 1e-4) - 1.0 / np.maximum(ybar, 1e-4))
    return e2, ds2 / den + s2 / (4.0 * n) * dinv + e2 * 2.0 ** -21   # + the f32 output


@pytest.mark.parametrize("variant", ["mega", "bvh", "wavefront"])
def test_noise_estimate_equals_the_formula_on_replayed_paths(be, variant):
    arrays, cams, w, h = _scene("config1")
    be.upload_scene(arrays)
    n = 8
    rep = _replay("config1", "default", "philox", 50, 0.0, 0, n)
    lin, _, _ = be.render(cams["default"], Backend.params(w, h, n, 50, seed=SEED, variant=variant, moments=True), want_rgb8=False)
    compare_paths(_pixels(rep), lin[:, :, None, :3], f"noise frame {variant}")
    err, _ = be.noise()
    rob = rep["robust"].all(axis=2)
    e2, bound = _err2_bound(rep["y"], rep["tol"], n)
    d = np.abs(err.astype(np.float64) ** 2 - e2)
    ratio = d / bound
    print(f"noise {variant}: {int(rob.sum())} robust pixels of {rob.size}, worst |e^2 - formula| / bound {ratio[rob].max():.3g}")
    bad = rob & ~(ratio <= 1.0)
    assert not bad.any(), (f"{int(bad.sum())} pixels: worst {np.unravel_index(np.argmax(np.where(bad, ratio, 0)), bad.shape)}, "
                           f"e {err[bad][:3]}, formula {np.sqrt(e2[bad][:3])}")
