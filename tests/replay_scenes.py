"""Scenes and comparisons shared by the path-replay tests (test_replay_cpu.py, test_replay_gpu.py): a path traced in f32 by
the product against the oracle's f64 replay of the same path (oracle Scene.replay)."""
import numpy as np

import oracle
import rayz_b200
from rayz_b200 import _abi as abi


def config1(w=317, h=178, glass_heavy=False):
    """randomBouncing seed 42 (config 1; glass_heavy: every random sphere dielectric) at an odd frame size: thin lens, moving
    spheres, the r = 1000 checker ground."""
    arrays = rayz_b200.random_bouncing(w, seed=42, glass_heavy=glass_heavy).pool.arrays()
    return arrays, rayz_b200.Camera.init(20.0, 10.0, 0.6, (13, 2, 3), (0, 0, 0), (0, 1, 0), h, w).rz


def all_materials():
    """The hand-built scene of test_gpu_parity.test_moving_spheres_and_all_materials_small_scene (moving diffuse, fuzzy metal,
    glass and a hollow bubble, all three diffuse methods) with a metal of fuzz > 1 (min(fuzz, 1) applies), a checker nested in a
    checker whose 1 / scale is not an f32 number (also the root texture of a fuzzy metal: the kernels' checker-of-two-solids
    shortcut with its split f64 1 / scale), and two cameras: the original thin-lens one and one inside a glass sphere."""
    pool = rayz_b200.MemPool()
    inner = pool.add_checker(0.3, pool.add_solid((0.8, 0.1, 0.1)), pool.add_solid((0.1, 0.7, 0.2)))
    ck = pool.add_checker(0.5, inner, pool.add_solid((0.9, 0.9, 0.8)))
    pool.add_sphere((0, -100.5, -1), 100, pool.add_diffuse(ck))
    pool.add_sphere((0, 0, -1.2), 0.5, pool.add_diffuse(pool.add_solid((0.7, 0.3, 0.3)), abi.DIFFUSE_UNIT_SPHERE_SURFACE), (0, 0.4, 0))
    pool.add_sphere((-1, 0, -1), 0.5, pool.add_dielectric(1.5))
    pool.add_sphere((-1, 0, -1), 0.4, pool.add_dielectric(1.0 / 1.5))
    pool.add_sphere((1, 0, -1), 0.5, pool.add_metallic(pool.add_solid((0.8, 0.6, 0.2)), 0.7))
    pool.add_sphere((0.3, 0.9, -1.5), 0.35, pool.add_diffuse(pool.add_solid((0.2, 0.8, 0.3)), abi.DIFFUSE_UNIT_SPHERE), (0.5, 0, 0))
    pool.add_sphere((2.0, 0.2, -2.5), 0.7, pool.add_metallic(pool.add_solid((0.9, 0.9, 0.9)), 0.0))
    pool.add_sphere((-2.2, 0.3, -2.2), 0.6, pool.add_metallic(pool.add_solid((0.7, 0.8, 0.9)), 1.7))
    pool.add_sphere((0.5, 0.6, 0.8), 0.9, pool.add_dielectric(1.5))                      # the second camera sits in here
    pool.add_sphere((-0.6, -0.3, 0.2), 0.2, pool.add_diffuse(ck), (0.0, 0.3, 0.2))
    pool.add_sphere((1.3, -0.1, 0.1), 0.4, pool.add_metallic(inner, 0.2))           # a checker of two solids as the root texture
    w, h = 203, 114
    cams = {"outside": rayz_b200.Camera.init(30.0, 3.4, 2.0, (-2, 2, 1), (0, 0, -1), (0, 1, 0), h, w).rz,
            "in_glass": rayz_b200.Camera.init(70.0, 2.0, 0.0, (0.5, 0.6, 0.8), (0, 0, -1), (0, 1, 0), h, w).rz}
    return pool.arrays(), cams, w, h


def metal_floor():
    """A fuzz-1 metal floor seen at a slant, with a diffuse, a glass and a fuzzy metal sphere on it: the scatter of the floor
    absorbs a large share of the paths (r.n <= 0), so that the ended_absorbed counter is large next to what fragile paths can
    move."""
    pool = rayz_b200.MemPool()
    pool.add_sphere((0, -100, 0), 100, pool.add_metallic(pool.add_solid((0.8, 0.8, 0.7)), 1.0))
    pool.add_sphere((-1.2, 0.5, 0), 0.5, pool.add_diffuse(pool.add_solid((0.6, 0.3, 0.2))))
    pool.add_sphere((0, 0.5, 0), 0.5, pool.add_dielectric(1.5))
    pool.add_sphere((1.2, 0.5, 0), 0.5, pool.add_metallic(pool.add_solid((0.7, 0.7, 0.9)), 0.3))
    w, h = 160, 90
    return pool.arrays(), rayz_b200.Camera.init(50.0, 5.0, 0.0, (0, 1.2, 5), (0, 0.3, 0), (0, 1, 0), h, w).rz, w, h


def compare_paths(rep, rgb, label, tol_scale=1.0, fragile_max=None):
    """rgb: [h, w, spp, 3] product radiance of the same paths.  Every robust path within its tolerance, no exception; prints
    paths, fragile fraction and the worst robust error relative to its tolerance.  Returns the worst ratio."""
    rob = rep["robust"]
    err = np.abs(np.asarray(rgb, np.float64) - rep["rgb"]).max(axis=-1)
    ratio = err / (rep["tol"] * tol_scale)
    worst = float(ratio[rob].max()) if rob.any() else 0.0
    frag = 1.0 - float(rob.mean())
    rel = err[rob] / np.maximum(rep["rgb"][rob].max(axis=-1), 1e-3) if rob.any() else np.zeros(1)
    print(f"{label}: {rob.size} paths, fragile {frag:.3%}, worst robust err / tol {worst:.3g}, robust err / radiance "
          f"median {np.median(rel):.2g} max {rel.max():.2g}")
    bad = rob & ~(ratio <= 1.0)
    if bad.any():
        i = tuple(np.argwhere(bad)[np.argmax(ratio[bad])])
        raise AssertionError(f"{label}: {int(bad.sum())} robust paths outside their tolerance; worst (row, col, sample) {i}: "
                             f"got {rgb[i]}, replay {rep['rgb'][i]}, tol {rep['tol'][i]:.3g}, segments {rep['segs'][i]}, "
                             f"end {rep['end'][i]}, hits {rep['hits'][i]}, event hash {int(rep['hash'][i]):#x}")
    if fragile_max is not None:
        assert frag <= fragile_max, f"{label}: fragile fraction {frag:.3%} above {fragile_max:.1%}"
    return worst


def count_stats(rep):
    """The replay's RzStats counters: paths, segments, hits per kind, ended_*."""
    ends = [int((rep["end"] == e).sum()) for e in (oracle.END_SKY, oracle.END_ABSORBED, oracle.END_DEPTH)]
    st = {"paths": rep["segs"].size, "segments": int(rep["segs"].sum()), "hits_diffuse": int(rep["hits"][..., 0].sum()),
          "hits_metallic": int(rep["hits"][..., 1].sum()), "hits_dielectric": int(rep["hits"][..., 2].sum()),
          "ended_sky": ends[0], "ended_absorbed": ends[1], "ended_depth": ends[2]}
    return st


def stat_slack(rep, depth):
    """Bound on |product - replay| per counter from the fragile paths alone: a fragile path agrees up to its first fragile
    segment and may do anything after it (at most depth segments in all, one end)."""
    fr = ~rep["robust"]
    fseg = np.maximum(rep["fseg"][fr], 0).astype(np.int64)
    after = np.maximum(rep["segs"][fr].astype(np.int64) - fseg, depth - fseg + 1)
    n = int(fr.sum())
    s = int(after.sum())
    return {"paths": 0, "segments": s, "hits_diffuse": s, "hits_metallic": s, "hits_dielectric": s,
            "ended_sky": n, "ended_absorbed": n, "ended_depth": n}
