"""ctypes front-end of the CPU oracle (oracle/rayz_oracle.cpp).

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs.  Never imported by rayz_b200/ (the product).

Scenes travel as a plain dict of numpy arrays whose keys are the field names of `RzScene`
(include/rayz_cuda.h), so the oracle and the CUDA backend consume the same bytes.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "_build", "librayz_oracle.so")

SCENE_FIELDS = (
    ("sphere_center", np.float64, 3), ("sphere_velocity", np.float64, 3), ("sphere_radius", np.float64, 1),
    ("sphere_material", np.uint32, 1),
    ("mat_kind", np.uint32, 1), ("mat_fuzz", np.float64, 1), ("mat_ior", np.float64, 1), ("mat_texture", np.uint32, 1),
    ("mat_method", np.uint32, 1),
    ("tex_kind", np.uint32, 1), ("tex_color", np.float64, 3), ("tex_scale", np.float64, 1), ("tex_even", np.uint32, 1),
    ("tex_odd", np.uint32, 1),
)
STAT_NAMES = ("paths", "segments", "sphere_tests", "node_tests", "hits_diffuse", "hits_metallic",
              "hits_dielectric", "ended_sky", "ended_absorbed", "ended_depth")


class OrcCamera(C.Structure):
    _fields_ = [("look_from", C.c_double * 3), ("px_du", C.c_double * 3), ("px_dv", C.c_double * 3),
                ("px_origin", C.c_double * 3), ("defocus_u", C.c_double * 3), ("defocus_v", C.c_double * 3),
                ("defocus", C.c_int32), ("reserved0", C.c_int32)]


def build(force: bool = False) -> str:
    """Compile the oracle with the committed Makefile; returns the .so path."""
    src = os.path.join(_HERE, "rayz_oracle.cpp")
    if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < os.path.getmtime(src):
        subprocess.run(["make", "-C", _HERE, "-s"], check=True)
    return _SO


_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(build())
        L = _lib
        dp, up = C.POINTER(C.c_double), C.POINTER(C.c_uint32)
        L.orc_scene_new.restype = C.c_void_p
        L.orc_scene_free.argtypes = [C.c_void_p]
        L.orc_scene_random_bouncing.restype = C.c_void_p
        L.orc_scene_random_bouncing.argtypes = [C.c_uint64, C.c_int32, C.c_int32, C.c_int32]
        L.orc_scene_counts.argtypes = [C.c_void_p, up, up, up]
        L.orc_scene_export.argtypes = [C.c_void_p] + [C.c_void_p] * 14
        L.orc_scene_from_arrays.restype = C.c_void_p
        L.orc_scene_from_arrays.argtypes = [C.c_uint32] * 3 + [C.c_void_p] * 14
        L.orc_camera_init.argtypes = [C.c_double] * 3 + [dp, dp, dp, C.c_uint64, C.c_uint64, C.POINTER(OrcCamera)]
        L.orc_get_ray.argtypes = [C.POINTER(OrcCamera), C.c_uint64, C.c_uint64, dp]
        L.orc_image_height.restype = C.c_uint64
        L.orc_image_height.argtypes = [C.c_uint64]
        L.orc_primary_ids.argtypes = [C.c_void_p, C.POINTER(OrcCamera), C.c_uint32, C.c_uint32, C.c_int32, C.c_void_p]
        L.orc_render.restype = C.c_uint64
        L.orc_render.argtypes = [C.c_void_p, C.POINTER(OrcCamera), C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32,
                                 C.c_uint64, C.c_uint32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]
        L.orc_quantise.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p]
        for name in ("orc_v3_dot",):
            getattr(L, name).restype = C.c_double
            getattr(L, name).argtypes = [dp, dp]
        L.orc_v3_mag.restype = C.c_double
        L.orc_v3_mag.argtypes = [dp]
        L.orc_v3_add.argtypes = [dp, dp, dp]
        L.orc_v3_mul.argtypes = [dp, C.c_double, dp]
        L.orc_v3_unit.argtypes = [dp, dp]
        L.orc_v3_amax.restype = C.c_int32
        L.orc_v3_amax.argtypes = [dp]
        for name in ("orc_clamp",):
            getattr(L, name).restype = C.c_double
            getattr(L, name).argtypes = [C.c_double] * 3
        for name in ("orc_min", "orc_max", "orc_reflectance"):
            getattr(L, name).restype = C.c_double
            getattr(L, name).argtypes = [C.c_double] * 2
        L.orc_refract.argtypes = [dp, dp, C.c_double, dp]
        L.orc_aabb_hit.restype = C.c_int32
        L.orc_aabb_hit.argtypes = [dp, dp, dp, dp, C.c_double, C.c_double]
        L.orc_aabb_enclose.argtypes = [dp] * 6
        L.orc_sphere_bbox.argtypes = [dp, dp, C.c_double, dp, dp]
        L.orc_sphere_hit.restype = C.c_int32
        L.orc_sphere_hit.argtypes = [dp, dp, C.c_double, dp, dp, C.c_double, C.c_double, C.c_double, dp]
        L.orc_texture_value.argtypes = [C.c_void_p, C.c_uint32, dp, dp]
        L.orc_sky.argtypes = [dp, dp]
        L.orc_rng_f64.argtypes = [C.c_uint64, C.c_uint32, C.c_void_p]
        L.orc_rng_u64.argtypes = [C.c_uint64, C.c_uint32, C.c_void_p]
        L.orc_bvh_export.restype = C.c_uint32
        L.orc_bvh_export.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p]
        L.orc_replay.argtypes = [C.c_void_p, C.POINTER(OrcCamera)] + [C.c_uint32] * 5 + [C.c_uint64, C.c_float, C.c_int32,
                                                                                       C.c_double, C.c_uint32] + [C.c_void_p] * 9
        L.orc_replay_uniforms.argtypes = [C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_int32, C.c_void_p]
    return _lib


def _d3(v):
    return (C.c_double * 3)(*[float(x) for x in v])


def v3(v):
    """numpy f64[3] -> ctypes pointer (kept alive by the returned array)."""
    a = np.ascontiguousarray(v, dtype=np.float64)
    return a, a.ctypes.data_as(C.POINTER(C.c_double))


class Scene:
    """Owns an oracle-side scene (MemPool restatement)."""

    def __init__(self, handle):
        self._h = C.c_void_p(handle)

    def __del__(self):
        try:
            if self._h:
                lib().orc_scene_free(self._h)
        except Exception:
            pass

    @staticmethod
    def random_bouncing(seed: int = 42, grid_lo: int = -11, grid_hi: int = 11, glass_heavy: bool = False) -> "Scene":
        """randomBouncing (rayz.zig:45-168) with an explicit seed."""
        return Scene(lib().orc_scene_random_bouncing(seed, grid_lo, grid_hi, int(glass_heavy)))

    @staticmethod
    def from_arrays(a: dict) -> "Scene":
        arrs = {}
        for name, dt, _ in SCENE_FIELDS:
            if name == "mat_method" and a.get(name) is None:
                arrs[name] = None
                continue
            arrs[name] = np.ascontiguousarray(a[name], dtype=dt)
        ns, nm, nt = len(arrs["sphere_radius"]), len(arrs["mat_kind"]), len(arrs["tex_kind"])
        ptrs = [arrs[n].ctypes.data if arrs[n] is not None else None for n, _, _ in SCENE_FIELDS]
        return Scene(lib().orc_scene_from_arrays(ns, nm, nt, *ptrs))

    def counts(self):
        ns, nm, nt = C.c_uint32(), C.c_uint32(), C.c_uint32()
        lib().orc_scene_counts(self._h, C.byref(ns), C.byref(nm), C.byref(nt))
        return ns.value, nm.value, nt.value

    def arrays(self) -> dict:
        ns, nm, nt = self.counts()
        n_of = {"sphere": ns, "mat": nm, "tex": nt}
        out = {}
        for name, dt, k in SCENE_FIELDS:
            n = n_of[name.split("_")[0]]
            out[name] = np.zeros((n, k) if k > 1 else (n,), dtype=dt)
        lib().orc_scene_export(self._h, *[out[n].ctypes.data for n, _, _ in SCENE_FIELDS])
        return out

    def primary_ids(self, cam: OrcCamera, w: int, h: int, use_bvh: bool = True) -> np.ndarray:
        out = np.empty((h, w), dtype=np.int32)
        lib().orc_primary_ids(self._h, C.byref(cam), w, h, int(use_bvh), out.ctypes.data)
        return out

    def render(self, cam: OrcCamera, w: int, h: int, spp: int, depth: int = 50, seed: int = 1, threads: int = 1,
               row_streams: bool = False, brute: bool = False, stats: bool = False):
        """Tracer.render (renderer.zig:72-101). Returns (linear f64 image [h,w,3], stats dict|None)."""
        out = np.empty((h, w, 3), dtype=np.float64)
        cnt = np.zeros(10, dtype=np.uint64) if stats else None
        n = lib().orc_render(self._h, C.byref(cam), w, h, spp, depth, seed, threads, int(row_streams), int(brute),
                             out.ctypes.data, cnt.ctypes.data if stats else None)
        assert n == w * h * spp
        return out, (dict(zip(STAT_NAMES, (int(x) for x in cnt))) if stats else None)

    def texture_value(self, tex: int, p) -> np.ndarray:
        o = np.zeros(3)
        pa, pp = v3(p)
        lib().orc_texture_value(self._h, tex, pp, o.ctypes.data_as(C.POINTER(C.c_double)))
        return o

    def replay(self, cam, w: int, h: int, sample_offset: int, spp: int, depth: int = 50, seed: int = 1, t_min: float = 0.0,
               sampler: str = "philox", perturb: float = 0.0, threads: int = 0) -> dict:
        """The backend's path algorithm replayed in f64 with the uniforms its kernels draw (rayz_oracle.cpp, namespace replay):
        one entry per path of samples [sample_offset, sample_offset + spp) of every pixel, arrays shaped [h, w, spp, ...].
        cam: an OrcCamera or the backend's RzCamera (same layout).  sampler: "philox", "sobol" or "sobol-rqmc".  perturb: the
        angle by which the perturbed replays turn every direction (0: the default, 1e-5 rad).
        Keys: rgb (clamped radiance), y (its luminance), segs, end (END_*), hits ([diffuse, metallic, dielectric]), hash (event
        sequence), reason / fseg (first fragile decision, REASONS; 0 = robust), robust, tol (radiance tolerance of a robust path)."""
        cam = cam if isinstance(cam, OrcCamera) else OrcCamera.from_buffer_copy(cam)
        n = (h, w, spp)
        out = dict(rgb=np.zeros(n + (3,)), y=np.zeros(n), segs=np.zeros(n, np.uint32), end=np.zeros(n, np.uint8),
                   hits=np.zeros(n + (3,), np.uint32), hash=np.zeros(n, np.uint64), reason=np.zeros(n, np.uint8),
                   fseg=np.zeros(n, np.int32), tol=np.zeros(n))
        lib().orc_replay(self._h, C.byref(cam), w, h, sample_offset, spp, depth, seed, t_min, SAMPLERS[sampler], perturb, threads,
                         *[out[k].ctypes.data for k in ("rgb", "y", "segs", "end", "hits", "hash", "reason", "fseg", "tol")])
        out["robust"] = out["reason"] == 0
        return out

    def bvh(self):
        ns, _, _ = self.counts()
        mx = 2 * ns + 2
        boxes = np.zeros((mx, 6)); links = np.zeros((mx, 4), dtype=np.int32); order = np.zeros(ns, dtype=np.uint32)
        n = lib().orc_bvh_export(self._h, mx, boxes.ctypes.data, links.ctypes.data, order.ctypes.data)
        return boxes[:n], links[:n], order


SAMPLERS = {"philox": 0, "sobol": 1, "sobol-rqmc": 2}
END_SKY, END_ABSORBED, END_DEPTH = 0, 1, 2
REASONS = ("robust", "tie", "graze", "t_min", "self_b", "diffuse_flip", "metal_rn", "tir", "fresnel", "self_out", "checker",
           "degenerate", "perturbed")


def replay_uniforms(seed: int, gpix: int, sample: int, depth: int, sampler: str = "philox") -> np.ndarray:
    """The uniforms the replay draws for one path: camera ux, uy, ut, ur, ua, then u.x..u.w of bounces 1..depth."""
    out = np.zeros(5 + 4 * depth)
    lib().orc_replay_uniforms(seed, gpix, sample, depth, SAMPLERS[sampler], out.ctypes.data)
    return out


def camera(vfov, focus_dist, defocus_angle, look_from, look_at, vup, img_h, img_w) -> OrcCamera:
    """Camera.init (camera.zig:18-57)."""
    cam = OrcCamera()
    lib().orc_camera_init(vfov, focus_dist, defocus_angle, _d3(look_from), _d3(look_at), _d3(vup), img_h, img_w,
                          C.byref(cam))
    return cam


def default_camera(img_w: int):
    """Camera of randomBouncing (rayz.zig:46-55) + Tracer.init's height (renderer.zig:39-40)."""
    h = int(lib().orc_image_height(img_w))
    return camera(20.0, 10.0, 0.6, (13, 2, 3), (0, 0, 0), (0, 1, 0), h, img_w), h


def get_ray(cam: OrcCamera, px: int, py: int):
    o = (C.c_double * 7)()
    lib().orc_get_ray(C.byref(cam), px, py, o)
    a = np.array(o[:])
    return a[0:3], a[3:6], a[6]


def quantise(rgb: np.ndarray) -> np.ndarray:
    """writePPM's per-pixel transform (image.zig:35-38)."""
    a = np.ascontiguousarray(rgb, dtype=np.float64).reshape(-1, 3)
    out = np.empty((a.shape[0], 3), dtype=np.uint8)
    lib().orc_quantise(a.ctypes.data, a.shape[0], out.ctypes.data)
    return out.reshape(rgb.shape)
