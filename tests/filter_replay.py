"""The pixel filters (include/rayz_cuda.h "RZ_RENDER_FILTER") restated in f64, shared by test_filter_cpu.py and
test_filter_gpu.py.

The exact normalised marginal CDF F of each filter, measured from the nearer edge of the support so that the tails are not
differences of near-equal numbers, and its inverse by bisection (filter_warp, to about 1e-12 px): the reference the library's
f32 warp rz_filter_warp is held to.  camera_rays restates the camera samples of a filtered render over the replay's own
uniforms (oracle.replay_uniforms), as mattes_replay.camera_rays does for the box, so that the first hits of a filtered frame
can be replayed in f64 (first_hits_robust)."""
import numpy as np
from scipy.special import erf, erfc

import mattes_replay
import oracle

BOX, TENT, GAUSSIAN, BLACKMAN_HARRIS = 0, 1, 2, 3
KINDS = {"box": BOX, "tent": TENT, "gaussian": GAUSSIAN, "blackman-harris": BLACKMAN_HARRIS}
DEFAULT_WIDTH = {BOX: 1.0, TENT: 2.0, GAUSSIAN: 3.0, BLACKMAN_HARRIS: 1.5}   # px
BH = (0.35875, 0.48829, 0.14128, 0.01168)
_C = 3.0 * np.sqrt(2.0)   # 1 / (s sqrt 2) of the unit-width Gaussian, s = 1/6


def _edge_mass(kind, d):
    """The unit-width filter's mass (not normalised) from its left edge to x = d - 1/2, d in [0, 1/2], and its total / 2."""
    d = np.asarray(d, np.float64)
    if kind == TENT:
        return d * d, 0.25
    if kind == GAUSSIAN:
        e = np.exp(-_C * _C / 4.0)
        k = np.sqrt(np.pi) / (2.0 * _C)
        return k * (erfc(_C * (0.5 - d)) - erfc(_C / 2.0)) - d * e, k * erf(_C / 2.0) - 0.5 * e
    if kind == BLACKMAN_HARRIS:
        a0, a1, a2, a3 = BH
        tp = 2.0 * np.pi
        return a0 * d - a1 / tp * np.sin(tp * d) + a2 / (2 * tp) * np.sin(2 * tp * d) - a3 / (3 * tp) * np.sin(3 * tp * d), a0 / 2
    return d, 0.5   # box


def density(kind, width, x):
    """The filter's marginal g at offset x px, not normalised (0 outside the support)."""
    x = np.asarray(x, np.float64) / width
    if kind == TENT:
        g = 1.0 - 2.0 * np.abs(x)
    elif kind == GAUSSIAN:
        g = np.exp(-_C * _C * x * x) - np.exp(-_C * _C / 4.0)
    elif kind == BLACKMAN_HARRIS:
        a0, a1, a2, a3 = BH
        g = a0 + a1 * np.cos(2 * np.pi * x) + a2 * np.cos(4 * np.pi * x) + a3 * np.cos(6 * np.pi * x)
    else:
        g = np.ones_like(x)
    return np.where(np.abs(x) <= 0.5, np.maximum(g, 0.0), 0.0)


def cdf(kind, width, x):
    """F(x): the normalised marginal's mass below offset x px, f64, from the nearer edge."""
    x = np.clip(np.asarray(x, np.float64) / width, -0.5, 0.5)
    m_lo, half = _edge_mass(kind, x + 0.5)
    m_hi, _ = _edge_mass(kind, 0.5 - x)
    return np.where(x <= 0.0, m_lo / (2.0 * half), 1.0 - m_hi / (2.0 * half))


def filter_warp(kind, width, u, iters=48):
    """The exact warp: the offset x px with F(x) = u, by bisection on the f64 CDF over the half nearer u's edge."""
    u = np.asarray(u, np.float64)
    v = np.minimum(u, 1.0 - u)
    _, half = _edge_mass(kind, 0.5)
    t = 2.0 * half * v
    lo, hi = np.zeros_like(v), np.full_like(v, 0.5)
    for _ in range(iters):
        m = 0.5 * (lo + hi)
        below = _edge_mass(kind, m)[0] < t
        lo, hi = np.where(below, m, lo), np.where(below, hi, m)
    x = width * (0.5 - 0.5 * (lo + hi))
    return np.where(u >= 0.5, x, -x)


def flags_of(pixel_filter, filter_width=None):
    """The RzRenderParams.flags field of a filter (RZ_RENDER_FILTER): kind name, width in px (None: the kind's default)."""
    w16 = 0 if filter_width is None else int(round(filter_width * 16))
    return (KINDS[pixel_filter] << 8) | (w16 << 16)


def camera_rays(cam, w, h, sample_offset, spp, seed, sampler="philox", pixel_filter="box", filter_width=None, rows=None):
    """Origins, unit directions and shutter times of the camera samples under a pixel filter, f64 over the replay's uniforms:
    [len(rows), w, spp, 3], [..., 3], [...].  The box gives mattes_replay.camera_rays' numbers bit for bit."""
    kind = KINDS[pixel_filter]
    width = DEFAULT_WIDTH[kind] if filter_width is None else filter_width
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
    if kind == BOX:
        x, y = i + (u[..., 0] - 0.5), j + (u[..., 1] - 0.5)
    else:
        x, y = i + filter_warp(kind, width, u[..., 0]), j + filter_warp(kind, width, u[..., 1])
    d = v["px_du"] * x[..., None] + v["px_dv"] * y[..., None] + v["px_origin"] - o
    d = d / np.sqrt((d * d).sum(axis=-1, keepdims=True))
    return o, d, u[..., 2]


def first_hits_robust(arrays, o, d, time, t_min=1e-4, margin=1e-4, chunk=256):
    """mattes_replay.first_hits with a robustness flag: (ids, robust).  A ray is robust when no sphere ahead of it passes
    within `margin` of its silhouette (| |l|^2 - r^2 | < margin r^2, |l| the ray line's distance from the centre) and its
    closest root is not within margin of another sphere's: an f32 ray within ~1e-6 rad of this one must hit the same sphere."""
    ids = mattes_replay.first_hits(arrays, o, d, time, t_min, chunk)
    shape = time.shape
    o, d, time = o.reshape(-1, 3), d.reshape(-1, 3), time.reshape(-1)
    c, v, r = arrays["sphere_center"], arrays["sphere_velocity"], arrays["sphere_radius"]
    robust = np.ones(len(time), bool)
    ts = np.full((len(time), 2), np.inf)
    for k0 in range(0, len(r), chunk):
        k1 = min(k0 + chunk, len(r))
        oc = c[None, k0:k1] + v[None, k0:k1] * time[:, None, None] - o[:, None]
        b = (oc * d[:, None]).sum(axis=-1)
        l = oc - d[:, None] * b[..., None]
        nd = (l * l).sum(axis=-1) - r[None, k0:k1] ** 2
        ahead = b + r[None, k0:k1] > t_min
        robust &= ~(ahead & (np.abs(nd) < margin * r[None, k0:k1] ** 2)).any(axis=1)
        sq = np.sqrt(np.where(nd < 0, -nd, np.nan))
        t = np.where(b - sq > t_min, b - sq, b + sq)
        t = np.where(t > t_min, t, np.inf)
        ts = np.sort(np.concatenate([ts, t], axis=1), axis=1)[:, :2]
    with np.errstate(invalid="ignore"):
        robust &= ~(np.isfinite(ts[:, 1]) & (ts[:, 1] - ts[:, 0] < margin * ts[:, 0]))
    return ids, robust.reshape(shape)
