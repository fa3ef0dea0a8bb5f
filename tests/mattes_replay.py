"""The first-hit id of every replayed camera sample (include/rayz_cuda.h "ID mattes"), shared by test_mattes_cpu.py and
test_mattes_gpu.py.

The oracle's replay (oracle Scene.replay) says whether a path's camera segment is robust (reason / fseg) and how many hits of
each material kind it made, but not which sphere it hit first.  Every uniform is a pure function of (seed, pixel, sample), so
the camera ray of a sample is restated here in f64 from the replay's own uniforms (oracle.replay_uniforms) and the replay's
camera formulas (rayz_oracle.cpp, replay::trace), and followed to its closest sphere over every sphere with the replay's root
rule.  A sample's first hit counts as proven when its depth-1 replay has no fragile decision in the camera segment: robust, or
a first fragile decision after it (fseg >= 1)."""
import numpy as np

import oracle


def camera_rays(cam, w, h, sample_offset, spp, seed, sampler="philox", rows=None):
    """Origins, unit directions and shutter times of the camera samples: [len(rows), w, spp, 3], [..., 3], [...]."""
    rows = range(h) if rows is None else rows
    v = {k: np.array(getattr(cam, k)[:], np.float64) for k in ("look_from", "px_du", "px_dv", "px_origin", "defocus_u", "defocus_v")}
    u = np.array([[[oracle.replay_uniforms(seed, j * w + i, sample_offset + s, 0, sampler)[:5] for s in range(spp)]
                   for i in range(w)] for j in rows])
    o = np.broadcast_to(v["look_from"], u.shape[:3] + (3,)).copy()
    if cam.defocus:
        rad, a = np.sqrt(u[..., 3]), (u[..., 4] - 0.5) * 6.283185307179586476925286766559
        o = o + v["defocus_u"] * (rad * np.cos(a))[..., None] + v["defocus_v"] * (rad * np.sin(a))[..., None]
    i = np.arange(w, dtype=np.float64)[None, :, None]
    j = np.array(list(rows), dtype=np.float64)[:, None, None]
    x, y = i + (u[..., 0] - 0.5), j + (u[..., 1] - 0.5)
    d = v["px_du"] * x[..., None] + v["px_dv"] * y[..., None] + v["px_origin"] - o
    d = d / np.sqrt((d * d).sum(axis=-1, keepdims=True))
    return o, d, u[..., 2]


def first_hits(arrays, o, d, time, t_min=0.0, chunk=256):
    """The caller's index of each ray's closest sphere (replay::trace's root rule, ties to the lower index), -1 for a miss."""
    t_min = float(np.float32(t_min)) if t_min > 0 else float(np.float32(1e-4))
    shape = time.shape
    o, d, time = o.reshape(-1, 3), d.reshape(-1, 3), time.reshape(-1)
    c, v, r = arrays["sphere_center"], arrays["sphere_velocity"], arrays["sphere_radius"]
    best_t = np.full(len(time), np.inf)
    best_k = np.full(len(time), -1, np.int32)
    for k0 in range(0, len(r), chunk):
        k1 = min(k0 + chunk, len(r))
        oc = c[None, k0:k1] + v[None, k0:k1] * time[:, None, None] - o[:, None]
        b = (oc * d[:, None]).sum(axis=-1)
        l = oc - d[:, None] * b[..., None]
        ll = np.sqrt((l * l).sum(axis=-1))
        nd = ll * ll - r[None, k0:k1] ** 2
        sq = np.sqrt(np.where(nd < 0, -nd, np.nan))
        t = b - sq
        t = np.where(t > t_min, t, b + sq)
        t = np.where(t > t_min, t, np.inf)   # NaN (no root) compares false: no hit
        kk = np.argmin(t, axis=1)
        tt = t[np.arange(len(t)), kk]
        better = tt < best_t
        best_t = np.where(better, tt, best_t)
        best_k = np.where(better, k0 + kk, best_k).astype(np.int32)
    return best_k.reshape(shape)


def replay_first(scene, arrays, cam, w, h, sample_offset, spp, seed, t_min=0.0, sampler="philox"):
    """(first [h, w, spp] int32: caller's index of each sample's first-hit sphere, -1 for a miss; proven [h, w, spp] bool;
    the depth-1 replay)."""
    one = scene.replay(cam, w, h, sample_offset, spp, 1, seed=seed, t_min=t_min, sampler=sampler)
    o, d, time = camera_rays(cam, w, h, sample_offset, spp, seed, sampler)
    first = first_hits(arrays, o, d, time, t_min)
    proven = (one["reason"] == 0) | (one["fseg"] >= 1)
    return first, proven, one


def histograms(first, n_ids):
    """[h, w, n_ids + 1] counts of each pixel's samples per id; column 0 is the miss (id -1), column k + 1 sphere k."""
    h, w, spp = first.shape
    out = np.zeros((h * w, n_ids + 1), np.int64)
    np.add.at(out, (np.repeat(np.arange(h * w), spp), first.reshape(-1) + 1), 1)
    return out.reshape(h, w, n_ids + 1)


def ranked(hist, ranks):
    """A histogram's ranks, count descending then id ascending: (ids [..., ranks] with -2 past the distinct ids, counts)."""
    ids = np.arange(hist.shape[-1]) - 1
    order = np.lexsort((np.broadcast_to(ids, hist.shape), -hist), axis=-1)[..., :ranks]
    cnt = np.take_along_axis(hist, order, axis=-1)
    return np.where(cnt > 0, order - 1, -2).astype(np.int32), cnt
