"""Host side above the C ABI: a mirror of the reference's host API for the hot path.

Same names, argument meaning and defaults as the Zig host so tests read like the reference's:

    Camera.init            camera.zig:18-57      -> Camera.init(...)  (fills RzCamera)
    MemPool                ecs.zig:22-70         -> MemPool.add_texture/add_material/add_sphere
    Tracer.init / render   renderer.zig:29-101   -> Tracer(...).render()  == the C-ABI call
    Image / writePPM       image.zig:4-41        -> Image.writePPM
    randomBouncing         rayz.zig:45-168       -> random_bouncing(img_w, seed)
    std.Random.DefaultPrng (Zig std)             -> Xoshiro256 (scene generation only)

Everything that touches pixels goes through librayz_cuda.so (rayz_b200._abi); nothing here
renders on the CPU.
"""
from __future__ import annotations

import ctypes as C
import math
import struct
from dataclasses import dataclass, field

import numpy as np

from . import _abi as abi

ASPECT_RATIO = 16.0 / 9.0  # renderer.zig:16
_M64 = (1 << 64) - 1


# ------------------------------------------------------------------------------- Zig std PRNG
class Xoshiro256:
    """std.Random.DefaultPrng: xoshiro256++ seeded through SplitMix64; float() == Random.float(f64)."""

    def __init__(self, seed: int):
        s = seed & _M64
        self.s = []
        for _ in range(4):
            s = (s + 0x9E3779B97F4A7C15) & _M64
            z = s
            z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & _M64
            z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & _M64
            self.s.append(z ^ (z >> 31))

    @staticmethod
    def _rotl(x, k):
        return ((x << k) | (x >> (64 - k))) & _M64

    def next(self) -> int:
        s = self.s
        r = (self._rotl((s[0] + s[3]) & _M64, 23) + s[0]) & _M64
        t = (s[1] << 17) & _M64
        s[2] ^= s[0]
        s[3] ^= s[1]
        s[1] ^= s[2]
        s[0] ^= s[3]
        s[2] ^= t
        s[3] = self._rotl(s[3], 45)
        return r

    def float(self) -> float:
        rand = self.next()
        lz = 64 - rand.bit_length()
        if lz >= 12:
            lz = 12
            while True:
                addl = 64 - self.next().bit_length()
                lz += addl
                if addl != 64:
                    break
                if lz >= 1022:
                    lz = 1022
                    break
        bits = ((1022 - lz) << 52) | (rand & 0xFFFFFFFFFFFFF)
        return struct.unpack("<d", struct.pack("<Q", bits))[0]

    def v3(self, low: float, high: float):
        """V3.random (vec.zig:9-16)."""
        scale = high - low
        return (self.float() * scale + low, self.float() * scale + low, self.float() * scale + low)


# ------------------------------------------------------------------------------- V3 helpers (f64, op order of vec.zig)
def _sub(a, b): return (a[0] - b[0], a[1] - b[1], a[2] - b[2])
def _add(a, b): return (a[0] + b[0], a[1] + b[1], a[2] + b[2])
def _mul(a, v): return (a[0] * v, a[1] * v, a[2] * v)
def _div(a, v): return _mul(a, 1 / v)                      # vec.zig:67-69: multiply by reciprocal
def _dot(a, b): return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]
def _mag(a): return math.sqrt(_dot(a, a))
def _unit(a): return _div(a, _mag(a))
def _cross(a, b): return (a[1] * b[2] - a[2] * b[1], a[2] * b[0] - a[0] * b[2], a[0] * b[1] - a[1] * b[0])


class Camera:
    """camera.zig:9-57.  `init` has the reference's 8-argument signature and fills an RzCamera."""

    DEG_TO_RAD = math.pi / 180.0

    def __init__(self, rz: abi.RzCamera):
        self.rz = rz

    @staticmethod
    def init(vfov, focus_dist, defocus_angle, look_from, look_at, vup, img_height: int, img_width: int) -> "Camera":
        fimg_h, fimg_w = float(img_height), float(img_width)
        vp_height = 2 * math.tan(vfov * Camera.DEG_TO_RAD / 2.0) * focus_dist
        vp_width = vp_height * fimg_w / fimg_h
        look_from = tuple(float(x) for x in look_from)
        w = _unit(_sub(look_from, tuple(float(x) for x in look_at)))
        u = _unit(_cross(tuple(float(x) for x in vup), w))
        v = _cross(w, u)
        vp_u = _mul(u, vp_width)
        vp_v = _mul(v, -vp_height)
        px_du = _div(vp_u, fimg_w)
        px_dv = _div(vp_v, fimg_h)
        defocus_radius = math.tan(defocus_angle * Camera.DEG_TO_RAD / 2) * focus_dist
        vp_origin = _add(_sub(_sub(_sub(look_from, _mul(w, focus_dist)), _div(vp_u, 2)), _div(vp_v, 2)),
                         _mul(_add(px_du, px_dv), 0.5))
        rz = abi.RzCamera()
        rz.look_from[:] = look_from
        rz.px_du[:] = px_du
        rz.px_dv[:] = px_dv
        rz.px_origin[:] = vp_origin
        rz.defocus_u[:] = _mul(u, defocus_radius)
        rz.defocus_v[:] = _mul(v, defocus_radius)
        rz.defocus = 1 if defocus_angle > 0 else 0
        return Camera(rz)


# ------------------------------------------------------------------------------- MemPool (ecs.zig:22-70)
@dataclass
class MemPool:
    """Three growable pools addressed by index handles; `arrays()` is the flatten the C ABI takes."""
    sphere_center: list = field(default_factory=list)
    sphere_velocity: list = field(default_factory=list)
    sphere_radius: list = field(default_factory=list)
    sphere_material: list = field(default_factory=list)
    mat_kind: list = field(default_factory=list)
    mat_fuzz: list = field(default_factory=list)
    mat_ior: list = field(default_factory=list)
    mat_texture: list = field(default_factory=list)
    mat_method: list = field(default_factory=list)
    tex_kind: list = field(default_factory=list)
    tex_color: list = field(default_factory=list)
    tex_scale: list = field(default_factory=list)
    tex_even: list = field(default_factory=list)
    tex_odd: list = field(default_factory=list)

    # addAndReturnHandle (ecs.zig:57-69): append, return index
    def add_solid(self, color) -> int:
        self.tex_kind.append(abi.TEX_SOLID); self.tex_color.append(tuple(float(c) for c in color))
        self.tex_scale.append(1.0); self.tex_even.append(0); self.tex_odd.append(0)
        return len(self.tex_kind) - 1

    def add_checker(self, scale: float, even: int, odd: int) -> int:
        self.tex_kind.append(abi.TEX_CHECKER); self.tex_color.append((0.0, 0.0, 0.0))
        self.tex_scale.append(float(scale)); self.tex_even.append(int(even)); self.tex_odd.append(int(odd))
        return len(self.tex_kind) - 1

    def add_diffuse(self, texture: int, method: int = abi.DIFFUSE_HEMISPHERE) -> int:
        return self._mat(abi.MAT_DIFFUSE, 0.0, 1.0, texture, method)

    def add_metallic(self, texture: int, fuzz: float = 0.0) -> int:
        return self._mat(abi.MAT_METALLIC, fuzz, 1.0, texture, abi.DIFFUSE_HEMISPHERE)

    def add_dielectric(self, refractive_index: float = 1.0) -> int:
        return self._mat(abi.MAT_DIELECTRIC, 0.0, refractive_index, 0, abi.DIFFUSE_HEMISPHERE)

    def _mat(self, kind, fuzz, ior, tex, method) -> int:
        self.mat_kind.append(kind); self.mat_fuzz.append(float(fuzz)); self.mat_ior.append(float(ior))
        self.mat_texture.append(int(tex)); self.mat_method.append(int(method))
        return len(self.mat_kind) - 1

    def add_sphere(self, center, radius: float, material: int, velocity=(0.0, 0.0, 0.0)) -> int:
        """Sphere{center: Ray{origin, dir}, radius, material} (geom.zig:11-14); velocity 0 == Sphere.stationary."""
        self.sphere_center.append(tuple(float(c) for c in center)); self.sphere_velocity.append(tuple(float(c) for c in velocity))
        self.sphere_radius.append(float(radius)); self.sphere_material.append(int(material))
        return len(self.sphere_radius) - 1

    def arrays(self) -> dict:
        f8 = lambda x, k: np.ascontiguousarray(np.asarray(x, dtype=np.float64).reshape((-1, k) if k > 1 else (-1,)))
        u4 = lambda x: np.ascontiguousarray(np.asarray(x, dtype=np.uint32).reshape(-1))
        return {"sphere_center": f8(self.sphere_center, 3), "sphere_velocity": f8(self.sphere_velocity, 3),
                "sphere_radius": f8(self.sphere_radius, 1), "sphere_material": u4(self.sphere_material),
                "mat_kind": u4(self.mat_kind), "mat_fuzz": f8(self.mat_fuzz, 1), "mat_ior": f8(self.mat_ior, 1),
                "mat_texture": u4(self.mat_texture), "mat_method": u4(self.mat_method),
                "tex_kind": u4(self.tex_kind), "tex_color": f8(self.tex_color, 3), "tex_scale": f8(self.tex_scale, 1),
                "tex_even": u4(self.tex_even), "tex_odd": u4(self.tex_odd)}


_F8 = ("sphere_center", "sphere_velocity", "sphere_radius", "mat_fuzz", "mat_ior", "tex_color", "tex_scale")
_U4 = ("sphere_material", "mat_kind", "mat_texture", "mat_method", "tex_kind", "tex_even", "tex_odd")


def scene_struct(arrays: dict):
    """dict of numpy arrays (RzScene field names) -> (RzScene, keepalive list)."""
    keep = {}
    sc = abi.RzScene()
    for k in _F8:
        keep[k] = np.ascontiguousarray(arrays[k], dtype=np.float64)
        setattr(sc, k, keep[k].ctypes.data_as(C.POINTER(C.c_double)))
    for k in _U4:
        if k == "mat_method" and arrays.get(k) is None:
            continue
        keep[k] = np.ascontiguousarray(arrays[k], dtype=np.uint32)
        setattr(sc, k, keep[k].ctypes.data_as(C.POINTER(C.c_uint32)))
    sc.n_spheres = keep["sphere_radius"].shape[0]
    sc.n_materials = keep["mat_kind"].shape[0]
    sc.n_textures = keep["tex_kind"].shape[0]
    return sc, keep


# ------------------------------------------------------------------------------- low-level backend handle
class Backend:
    """Owns one RzContext (include/rayz_cuda.h)."""

    BVH_BUILD = {"auto": 0, "host": 1, "device": 2}   # RZ_CFG_BVH_BUILD_* (include/rayz_cuda.h)

    def __init__(self, devices=(0,), bvh_build: str = "auto"):
        self.lib = abi.load()
        cfg = abi.RzConfig()
        cfg.flags = self.BVH_BUILD[bvh_build]
        cfg.n_devices = len(devices)
        for i, d in enumerate(devices):
            cfg.device_ids[i] = int(d)
        h = C.c_void_p()
        abi.check(self.lib.rayz_cuda_create(C.byref(cfg), C.byref(h)))
        self._h = h
        self.devices = tuple(devices)
        self._acc_shape = None   # (height, width, shard_index, shard_count, band_rows) of the last successful render: noise()'s rows

    def close(self):
        if getattr(self, "_h", None):
            self.lib.rayz_cuda_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_stream(self, cuda_stream: int | None):
        abi.check(self.lib.rayz_cuda_set_stream(self._h, C.c_void_p(cuda_stream or 0)))

    def get_tuning(self) -> dict:
        t = abi.RzTuning()
        abi.check(self.lib.rayz_cuda_get_tuning(self._h, C.byref(t)))
        return t.as_dict()

    def set_tuning(self, rays_per_thread: int = 0, chunk: int = 0, **fields):
        """rayz_cuda_get_tuning -> change -> rayz_cuda_set_tuning (include/rayz_cuda.h: RzTuning).  `chunk` sets the work-unit
        size of the persistent kernels and of the primary kernel alike; other fields by name, e.g. second_stages=3."""
        t = abi.RzTuning()
        abi.check(self.lib.rayz_cuda_get_tuning(self._h, C.byref(t)))
        if rays_per_thread:
            t.rays_per_thread = rays_per_thread
        if chunk:
            t.chunk = t.chunk_primary = chunk
        for k, v in fields.items():
            if k not in dict(abi.RzTuning._fields_):
                raise KeyError(k)
            setattr(t, k, v)
        abi.check(self.lib.rayz_cuda_set_tuning(self._h, C.byref(t)))

    def debug_sort_keys(self, keys: np.ndarray):
        """Test hook: the staged K1's key sort (rz_sort.cu) on caller-supplied 16-bit keys -> (keys in slot order, output word in slot order:
        entry index | reach class << 28)."""
        keys = np.ascontiguousarray(keys, dtype=np.uint16)
        ko = np.empty_like(keys)
        io = np.empty(keys.shape, dtype=np.uint32)
        abi.check(self.lib.rayz_cuda_debug_sort_keys(self._h, keys.ctypes.data, keys.size, ko.ctypes.data, io.ctypes.data))
        return ko, io

    def upload_scene(self, arrays: dict):
        sc, keep = scene_struct(arrays)
        abi.check(self.lib.rayz_cuda_upload_scene(self._h, C.byref(sc)))
        self.scene_bytes = sum(a.nbytes for a in keep.values())

    @staticmethod
    def params(width, height, spp, max_depth=50, seed=1, sample_offset=0, variant="auto", t_min=0.0, shard_index=0,
               shard_count=1, band_rows=0, collect_stats=False, serial_passes=False, accumulate=False,
               moments=False, sobol=False, rqmc=False, passes=False, pixel_filter="box", filter_width=None) -> abi.RzRenderParams:
        """RzRenderParams.  accumulate: add this batch to the previous render's sums (RZ_RENDER_ACCUMULATE; sample_offset must
        continue where they end); moments: also sum each path's luminance squared, so that noise() can estimate the error;
        sobol: draw the camera and scatter samples from Owen-scrambled Sobol pairs instead of Philox (RZ_RENDER_SOBOL);
        rqmc: two independently scrambled Sobol replicates per pixel, so that the noise estimate sees the stratification
        (RZ_RENDER_RQMC).  rqmc does not imply sobol or moments: the library refuses it without both, and with an odd spp or
        sample_offset.  passes: also sum each path's radiance into its light-path pass, so that passes() can split the frame
        (RZ_RENDER_PASSES; no pixel changes).  pixel_filter: the reconstruction filter each camera sample's offset is drawn
        from, "box" (the default: the reference's uniform jitter), "tent", "gaussian" or "blackman-harris" (RZ_RENDER_FILTER);
        filter_width: its full width in px, None for the kind's default (2, 3 and 1.5 px), else 1 to 4 px in steps of 1/16
        (a width with the box is refused by the library)."""
        if pixel_filter not in abi.FILTERS:
            raise ValueError(f"pixel_filter must be one of {sorted(abi.FILTERS)}, not {pixel_filter!r}")
        w16 = 0
        if filter_width is not None:
            w16 = int(round(float(filter_width) * 16))
            if w16 != float(filter_width) * 16 or not 0 <= w16 <= 255:
                raise ValueError(f"filter_width must be a multiple of 1/16 px, not {filter_width!r}")
        p = abi.RzRenderParams()
        p.width, p.height, p.spp, p.max_depth = width, height, spp, max_depth
        p.seed, p.sample_offset = seed, sample_offset
        p.variant = abi.VARIANTS[variant] if isinstance(variant, str) else int(variant)
        p.t_min = t_min
        p.shard_index, p.shard_count, p.band_rows = shard_index, shard_count, band_rows
        p.collect_stats = 1 if collect_stats else 0
        p.flags = ((abi.RENDER_SERIAL_PASSES if serial_passes else 0) | (abi.RENDER_ACCUMULATE if accumulate else 0)
                   | (abi.RENDER_MOMENTS if moments else 0) | (abi.RENDER_SOBOL if sobol else 0) | (abi.RENDER_RQMC if rqmc else 0)
                   | (abi.RENDER_PASSES if passes else 0) | abi.render_filter(abi.FILTERS[pixel_filter], w16))
        return p

    def reserve(self, p: abi.RzRenderParams):
        """rayz_cuda_reserve: allocate the per-render device buffers ahead of the first render."""
        abi.check(self.lib.rayz_cuda_reserve(self._h, C.byref(p)))

    def shard_rows(self, p: abi.RzRenderParams) -> int:
        return int(self.lib.rayz_cuda_context_rows(self._h, p.height, p.shard_index, p.shard_count, p.band_rows))

    def render(self, cam: abi.RzCamera, p: abi.RzRenderParams, want_linear=True, want_rgb8=True,
               out_linear: np.ndarray | None = None, out_rgb8: np.ndarray | None = None):
        """rayz_cuda_render: host buffers, H2D/D2H inside. Returns (linear [rows,w,4] f32, rgb8 [rows,w,3] u8, paths)."""
        rows = self.shard_rows(p)
        if want_linear and out_linear is None:
            out_linear = np.empty((rows, p.width, 4), dtype=np.float32)
        if want_rgb8 and out_rgb8 is None:
            out_rgb8 = np.empty((rows, p.width, 3), dtype=np.uint8)
        n = C.c_uint64()
        abi.check(self.lib.rayz_cuda_render(self._h, C.byref(cam), C.byref(p),
                                            out_linear.ctypes.data if want_linear else None,
                                            out_rgb8.ctypes.data if want_rgb8 else None, C.byref(n)))
        self._acc_shape = (p.height, p.width, p.shard_index, p.shard_count, p.band_rows)
        return (out_linear if want_linear else None), (out_rgb8 if want_rgb8 else None), n.value

    def render_device(self, cam: abi.RzCamera, p: abi.RzRenderParams, sync=True):
        """rayz_cuda_render_device: results stay in HBM. Returns (d_linear ptr, d_rgb8 ptr, paths)."""
        dl, d8, n = C.c_void_p(), C.c_void_p(), C.c_uint64()
        abi.check(self.lib.rayz_cuda_render_device(self._h, C.byref(cam), C.byref(p), C.byref(dl), C.byref(d8), C.byref(n),
                                                   1 if sync else 0))
        self._acc_shape = (p.height, p.width, p.shard_index, p.shard_count, p.band_rows)
        return dl.value, d8.value, n.value

    def noise(self, target: float = 0.0):
        """rayz_cuda_noise: per-pixel standard error of the displayed value of the accumulated frame (needs moments=True) ->
        (err [rows,w] f32, summary dict: samples, n_pixels, n_above (pixels with err > target), mean_err, rms_err, max_err)."""
        nz = abi.RzNoise()
        if self._acc_shape is None:   # nothing rendered: the library says why
            abi.check(self.lib.rayz_cuda_noise(self._h, float(target), None, C.byref(nz)))
        rows, w = int(self.lib.rayz_cuda_context_rows(self._h, self._acc_shape[0], *self._acc_shape[2:])), self._acc_shape[1]
        err = np.empty((rows, w), dtype=np.float32)
        abi.check(self.lib.rayz_cuda_noise(self._h, float(target), err.ctypes.data, C.byref(nz)))
        return err, nz.as_dict()

    def render_to_noise(self, cam: abi.RzCamera, p: abi.RzRenderParams, target: float, max_spp: int, want_linear=True,
                        want_rgb8=True, adaptive=False, pooled=False):
        """rayz_cuda_render_to_noise: p.spp samples, then batches doubling the count until rms_err <= target or max_spp.
        adaptive (RZ_RENDER_ADAPTIVE): the same schedule per pixel, until every pixel's error is <= target or max_spp; the
        per-pixel counts are then pixel_samples().  pooled (RZ_RENDER_ADAPTIVE_POOLED): each pixel's error is pooled with its
        row segment's, so that the per-pixel bound holds for the measured error, not only for the estimate; the library
        refuses it without adaptive.  Returns (linear [rows,w,4] f32, rgb8 [rows,w,3] u8, paths, summary dict as noise())."""
        if adaptive or pooled:
            p = abi.RzRenderParams.from_buffer_copy(p)
            p.flags |= (abi.RENDER_ADAPTIVE if adaptive else 0) | (abi.RENDER_ADAPTIVE_POOLED if pooled else 0)
        rows = self.shard_rows(p)
        lin = np.empty((rows, p.width, 4), dtype=np.float32) if want_linear else None
        rgb8 = np.empty((rows, p.width, 3), dtype=np.uint8) if want_rgb8 else None
        n, nz = C.c_uint64(), abi.RzNoise()
        abi.check(self.lib.rayz_cuda_render_to_noise(self._h, C.byref(cam), C.byref(p), float(target), int(max_spp),
                                                     lin.ctypes.data if want_linear else None,
                                                     rgb8.ctypes.data if want_rgb8 else None, C.byref(n), C.byref(nz)))
        self._acc_shape = (p.height, p.width, p.shard_index, p.shard_count, p.band_rows)
        return lin, rgb8, n.value, nz.as_dict()

    def pixel_samples(self) -> np.ndarray:
        """rayz_cuda_pixel_samples: every pixel's sample count of the accumulated frame -> [rows,w] u32 (uniform after a
        plain render or batches, each pixel's own after render_to_noise(adaptive=True))."""
        if self._acc_shape is None:   # nothing rendered: the library says why
            abi.check(self.lib.rayz_cuda_pixel_samples(self._h, None))
        rows, w = int(self.lib.rayz_cuda_context_rows(self._h, self._acc_shape[0], *self._acc_shape[2:])), self._acc_shape[1]
        out = np.empty((rows, w), dtype=np.uint32)
        abi.check(self.lib.rayz_cuda_pixel_samples(self._h, out.ctypes.data))
        return out

    def passes(self) -> np.ndarray:
        """rayz_cuda_passes: the light-path passes of the accumulated frame (rendered with passes=True) -> [7,rows,w,4] f32,
        plane i = pass abi.PASS_NAMES[i], each laid out like render()'s linear; they sum to the linear frame to f32 rounding."""
        if self._acc_shape is None:   # nothing rendered: the library says why
            abi.check(self.lib.rayz_cuda_passes(self._h, None))
        rows, w = int(self.lib.rayz_cuda_context_rows(self._h, self._acc_shape[0], *self._acc_shape[2:])), self._acc_shape[1]
        out = np.empty((abi.PASS_COUNT, rows, w, 4), dtype=np.float32)
        abi.check(self.lib.rayz_cuda_passes(self._h, out.ctypes.data))
        return out

    def guides(self, cam: abi.RzCamera, p: abi.RzRenderParams):
        """rayz_cuda_render_guides: the first hits of the camera samples a render with these parameters traces ->
        (albedo [rows,w,4] f32: rgb mean albedo, a coverage; normal [rows,w,4] f32: xyz mean unit normal, w mean hit distance).
        Leaves the accumulated frame, stats and timing as they were."""
        rows = self.shard_rows(p)
        albedo = np.empty((rows, p.width, 4), dtype=np.float32)
        normal = np.empty((rows, p.width, 4), dtype=np.float32)
        abi.check(self.lib.rayz_cuda_render_guides(self._h, C.byref(cam), C.byref(p), albedo.ctypes.data, normal.ctypes.data))
        return albedo, normal

    def mattes(self, cam: abi.RzCamera, p: abi.RzRenderParams, ranks: int = 6):
        """rayz_cuda_render_mattes: the first-hit ids of the camera samples a render with these parameters traces, ranked per
        pixel by count descending, then id ascending -> (ids [rows,w,ranks] int32: caller's sphere index, abi.MATTE_MISS for the
        sky, abi.MATTE_EMPTY past the pixel's distinct ids; coverage [rows,w,ranks] f32: count / spp).  Leaves the accumulated
        frame, the guides, stats and timing as they were."""
        rows = self.shard_rows(p)
        ids = np.empty((rows, p.width, max(int(ranks), 1)), dtype=np.int32)
        cov = np.empty(ids.shape, dtype=np.float32)
        abi.check(self.lib.rayz_cuda_render_mattes(self._h, C.byref(cam), C.byref(p), ranks, ids.ctypes.data, cov.ctypes.data))
        return ids, cov

    def denoise(self, iterations: int = 5, sigma_luminance: float = 4.0, sigma_normal: float = 128.0, sigma_depth: float = 1.0):
        """rayz_cuda_denoise: the accumulated frame (needs moments=True) filtered by the edge-avoiding à-trous filter, steered by
        its noise estimate and the guides of the last guides() call of the same frame, camera and seed ->
        (linear [rows,w,4] f32, rgb8 [rows,w,3] u8).  iterations=0 returns the resolved frame.  Leaves the accumulated frame,
        stats and timing as they were."""
        dp = abi.RzDenoiseParams()
        dp.struct_size = C.sizeof(abi.RzDenoiseParams)
        dp.iterations = iterations
        dp.sigma_luminance, dp.sigma_normal, dp.sigma_depth = sigma_luminance, sigma_normal, sigma_depth
        if self._acc_shape is None:   # nothing rendered: the library says why
            abi.check(self.lib.rayz_cuda_denoise(self._h, C.byref(dp), None, None))
        rows, w = int(self.lib.rayz_cuda_context_rows(self._h, self._acc_shape[0], *self._acc_shape[2:])), self._acc_shape[1]
        lin = np.empty((rows, w, 4), dtype=np.float32)
        rgb8 = np.empty((rows, w, 3), dtype=np.uint8)
        abi.check(self.lib.rayz_cuda_denoise(self._h, C.byref(dp), lin.ctypes.data, rgb8.ctypes.data))
        return lin, rgb8

    def primary_ids(self, cam: abi.RzCamera, width: int, height: int, use_bvh=True) -> np.ndarray:
        out = np.empty((height, width), dtype=np.int32)
        abi.check(self.lib.rayz_cuda_primary_ids(self._h, C.byref(cam), width, height, 1 if use_bvh else 0, out.ctypes.data))
        return out

    def stage_stats(self, stage: int) -> dict:
        """Counters of one stage of the staged K1: 0 primary kernel, 1 sorted stages, 2 persistent tail kernel (BVH, or the brute-force megakernel)."""
        s = abi.RzStats()
        abi.check(self.lib.rayz_cuda_stage_stats(self._h, stage, C.byref(s)))
        return s.as_dict()

    def stats(self) -> dict:
        s = abi.RzStats()
        abi.check(self.lib.rayz_cuda_stats(self._h, C.byref(s)))
        return s.as_dict()

    def timing(self) -> dict:
        t = abi.RzTiming()
        abi.check(self.lib.rayz_cuda_timing(self._h, C.byref(t)))
        return t.as_dict()

    def fp32_peak(self, millis=200):
        tf, sms = C.c_double(), C.c_int32()
        abi.check(self.lib.rayz_cuda_fp32_peak(self._h, millis, C.byref(tf), C.byref(sms)))
        return tf.value, sms.value


# ------------------------------------------------------------------------------- Image (image.zig)
class Image:
    """image.zig:4-41: linear f64 RGB framebuffer `pixels[j*w+i]`; writePPM writes ASCII P3."""

    def __init__(self, h: int, w: int):
        self.h, self.w = h, w
        self.pixels = np.zeros((h * w, 3), dtype=np.float64)
        self.rgb8 = None  # filled by Tracer.render: the device-side sqrt/clamp/trunc of image.zig:35-38

    def writePPM(self, f):
        if self.rgb8 is None:
            raise RuntimeError("Image.writePPM: no rendered pixels (call Tracer.render first)")
        f.write(f"P3\n{self.w} {self.h}\n255\n")
        q = self.rgb8.reshape(-1, 3)
        f.write("\n".join(f"{a} {b} {c}" for a, b, c in q.tolist()))
        f.write("\n")


# ------------------------------------------------------------------------------- Tracer (renderer.zig)
class Tracer:
    """renderer.zig:18-101.  `render()` is the drop-in: it returns the number of primary rays
    (`!usize`, :72,100) and fills `img.pixels`; the pixel loop itself runs on the GPU."""

    def __init__(self, img_w: int, vfov, focus_dist, defocus_angle, look_from, look_at, vup, devices=(0,), seed: int = 1):
        height = int(float(img_w) / ASPECT_RATIO)  # renderer.zig:39-40
        self.camera = Camera.init(vfov, focus_dist, defocus_angle, look_from, look_at, vup, height, img_w)
        self.img = Image(height, img_w)
        self.max_bounces = 50      # renderer.zig:23
        self.samples_per_px = 10   # renderer.zig:24
        self.pool = MemPool()
        self.seed = seed           # the reference seeds from the OS (renderer.zig:55-59)
        self.variant = "auto"
        self.pixel_filter = "box"  # reconstruction filter of render(), render_guides(), render_mattes() and so denoise():
        self.filter_width = None   # "tent", "gaussian" or "blackman-harris", width in px (None: the kind's default)
        self.sampler = "philox"    # or "sobol": low-discrepancy camera and scatter samples (RZ_RENDER_SOBOL) in render(),
                                   # render_guides() and so the denoised frame; or "sobol-rqmc": the same with two replicates
                                   # per pixel and the noise estimate they allow (RZ_RENDER_RQMC, with moments)
        self.devices = devices
        self.noise = None          # summary of the last render(noise_target=...) (rayz_cuda_render_to_noise)
        self.pixel_samples = None  # [h, w] per-pixel sample counts of the last render(noise_target=..., adaptive=True)
        self.albedo = None         # [h, w, 4] guide buffers of the last render_guides(): rgb albedo + coverage
        self.normal = None         # [h, w, 4] ... unit normal + hit distance
        self.denoised = None       # (linear [h, w, 4], rgb8 [h, w, 3]) of the last denoise()
        self.matte_ids = None      # [h, w, ranks] ID mattes of the last render_mattes(): caller's sphere indices by rank
        self.matte_coverage = None  # [h, w, ranks] ... the fraction of the pixel's samples each covers
        self._backend = None
        self._uploaded = None      # the pool arrays of the backend's last scene upload

    SAMPLERS = {"philox": {}, "sobol": {"sobol": True}, "sobol-rqmc": {"sobol": True, "rqmc": True, "moments": True}}

    def _sampler(self) -> dict:
        """Backend.params keywords of self.sampler."""
        if self.sampler not in self.SAMPLERS:
            raise ValueError(f"Tracer.sampler must be 'philox', 'sobol' or 'sobol-rqmc', not {self.sampler!r}")
        return dict(self.SAMPLERS[self.sampler])

    def _filter(self) -> dict:
        """Backend.params keywords of the pixel filter."""
        return {"pixel_filter": self.pixel_filter, "filter_width": self.filter_width}

    @property
    def backend(self) -> Backend:
        if self._backend is None:
            self._backend = Backend(self.devices)
        return self._backend

    def render(self, noise_target: float | None = None, max_spp: int = 4096, adaptive: bool = False, moments: bool = False,
               pooled: bool = False, passes: bool = False) -> int:
        """noise_target (displayed-value rms error, 1/255 = one 8-bit step): start at samples_per_px and double the samples
        until the frame's rms error reaches it or max_spp samples are in (rayz_cuda_render_to_noise); `self.noise` then holds
        the summary.  adaptive: the target bounds every pixel's error, and only the pixels still above it get more samples;
        `self.pixel_samples` then holds the counts; pooled (with adaptive): each pixel stops on an error pooled with its row
        segment's (RZ_RENDER_ADAPTIVE_POOLED), so that the bound holds for the measured error; the library refuses it
        elsewhere.  Without a target, one render of samples_per_px, as the reference; moments: also sum what the per-pixel
        noise estimate needs (RZ_RENDER_MOMENTS, no pixel changes), so that denoise() can follow; passes: also sum the
        light-path passes (RZ_RENDER_PASSES, no pixel changes), so that passes() can follow."""
        b = self.backend
        arrays = self.pool.arrays()
        self._uploaded = None
        b.upload_scene(arrays)  # initHittables + bvh.build (renderer.zig:76-78)
        self._uploaded = arrays
        kw = self._sampler()
        kw["moments"] = moments or kw.get("moments", False)
        p = Backend.params(self.img.w, self.img.h, self.samples_per_px, self.max_bounces, self.seed, variant=self.variant, **kw,
                           **self._filter())
        if pooled:
            p.flags |= abi.RENDER_ADAPTIVE_POOLED
        if passes:
            p.flags |= abi.RENDER_PASSES
        if noise_target is None:
            lin, rgb8, rays = b.render(self.camera.rz, p)
        else:
            lin, rgb8, rays, self.noise = b.render_to_noise(self.camera.rz, p, noise_target, max_spp, adaptive=adaptive)
            self.pixel_samples = b.pixel_samples() if adaptive else None
        self.img.pixels[:] = lin.reshape(-1, 4)[:, :3]
        self.img.rgb8 = rgb8
        return rays

    def passes(self) -> dict:
        """The light-path passes of the last render(passes=True) (rayz_cuda_passes): pass name (abi.PASS_NAMES) -> linear
        [h, w, 4] f32 image; the images sum to the render's linear frame to f32 rounding."""
        planes = self.backend.passes()
        return {name: planes[i] for i, name in enumerate(abi.PASS_NAMES)}

    def render_guides(self):
        """Guide buffers for a denoiser over the camera samples render() traces (samples_per_px, seed): first-hit albedo with
        coverage, and normal with hit distance (rayz_cuda_render_guides).  Returns (albedo, normal), also kept as
        self.albedo and self.normal.  The scene is uploaded only when the pool differs from the one this tracer last uploaded,
        so that the frame of a previous render() stays accumulated for denoise() (it used to be uploaded on every call, which
        ended that frame).  An upload made directly through self.backend is not seen: call render() after one."""
        b = self._backend_with_scene()
        self.albedo, self.normal = b.guides(self.camera.rz, self._first_hit_params())
        return self.albedo, self.normal

    def render_mattes(self, ranks: int = 6):
        """ID mattes over the camera samples render() traces (samples_per_px, seed, at most 1024): per pixel, the caller's
        indices of the spheres its samples hit first, ranked by coverage (rayz_cuda_render_mattes).  Returns (ids [h, w, ranks]
        int32, coverage [h, w, ranks] f32), also kept as self.matte_ids and self.matte_coverage.  The scene is uploaded as
        render_guides() uploads it: only when the pool changed."""
        b = self._backend_with_scene()
        self.matte_ids, self.matte_coverage = b.mattes(self.camera.rz, self._first_hit_params(), ranks)
        return self.matte_ids, self.matte_coverage

    def _backend_with_scene(self) -> Backend:
        """The backend, with the pool uploaded unless it equals the one this tracer last uploaded."""
        b = self.backend
        arrays = self.pool.arrays()
        # the scene render() uploaded stays: uploading it again would end the accumulated frame that denoise() filters
        if self._uploaded is None or arrays.keys() != self._uploaded.keys() or \
                not all(np.array_equal(arrays[k], self._uploaded[k]) for k in arrays):
            self._uploaded = None
            b.upload_scene(arrays)
            self._uploaded = arrays
        return b

    def _first_hit_params(self) -> abi.RzRenderParams:
        """The parameters of render()'s camera samples, for the first-hit calls (guides, mattes)."""
        return Backend.params(self.img.w, self.img.h, self.samples_per_px, self.max_bounces, self.seed, variant=self.variant,
                              **self._sampler(), **self._filter())

    def denoise(self, iterations: int = 5, sigma_luminance: float = 4.0, sigma_normal: float = 128.0, sigma_depth: float = 1.0):
        """The frame of the last render() (with moments=True, or a noise target) denoised with the guides of render_guides(),
        called after it (rayz_cuda_denoise).  Returns (linear [h,w,4] f32, rgb8 [h,w,3] u8), also kept as self.denoised."""
        self.denoised = self.backend.denoise(iterations, sigma_luminance, sigma_normal, sigma_depth)
        return self.denoised


# ------------------------------------------------------------------------------- scenes (rayz.zig)
def random_bouncing(img_w: int, seed: int = 42, grid_lo: int = -11, grid_hi: int = 11, glass_heavy: bool = False,
                    devices=(0,)) -> Tracer:
    """randomBouncing (rayz.zig:45-168) with an explicit scene seed.

    grid_lo/grid_hi widen the `a`,`b` loops (reference: -11..11; BASELINE config 4 uses -158..158);
    glass_heavy (config 5) makes every random sphere and the two non-glass big spheres dielectric
    (ior 1.5) while consuming the same PRNG draws, so sphere positions match the default scene.
    """
    tracer = Tracer(img_w, 20.0, 10.0, 0.6, (13, 2, 3), (0, 0, 0), (0, 1, 0), devices=devices)
    pool = tracer.pool
    rng = Xoshiro256(seed)
    # ground (:57-73): even, odd, checker, material, sphere
    te = pool.add_solid((0.2, 0.3, 0.1))
    to = pool.add_solid((0.9, 0.9, 0.9))
    tc = pool.add_checker(0.32, te, to)
    pool.add_sphere((0, -1000, 0), 1000, pool.add_diffuse(tc))
    # main three (:76-104)
    pool.add_sphere((0, 1, 0), 1.0, pool.add_dielectric(1.5))
    if glass_heavy:
        pool.add_sphere((-4, 1, 0), 1.0, pool.add_dielectric(1.5))
        pool.add_sphere((4, 1, 0), 1.0, pool.add_dielectric(1.5))
    else:
        pool.add_sphere((-4, 1, 0), 1.0, pool.add_diffuse(pool.add_solid((0.4, 0.2, 0.1))))
        pool.add_sphere((4, 1, 0), 1.0, pool.add_metallic(pool.add_solid((0.7, 0.6, 0.5)), 0.0))
    # randoms (:108-166)
    for a in range(grid_lo, grid_hi):
        for b in range(grid_lo, grid_hi):
            rand_mat = rng.float()
            center = (float(a) + 0.9 * rng.float(), 0.2, float(b) + 0.9 * rng.float())
            if _mag(_sub(center, (4.0, 0.2, 0.0))) <= 0.9:
                continue
            vel = (0.0, 0.0, 0.0)
            if rand_mat < 0.8:
                c1 = rng.v3(0, 1.0)
                c2 = rng.v3(0, 1.0)
                vy = rng.float() * 0.5
                if glass_heavy:
                    m = pool.add_dielectric(1.5)
                else:
                    m = pool.add_diffuse(pool.add_solid((c1[0] * c2[0], c1[1] * c2[1], c1[2] * c2[2])))
                    vel = _mul((0.0, 1.0, 0.0), vy)
            elif rand_mat < 0.95:
                fuzz = rng.float() * 0.5
                col = rng.v3(0.5, 1.0)
                m = pool.add_dielectric(1.5) if glass_heavy else pool.add_metallic(pool.add_solid(col), fuzz)
            else:
                m = pool.add_dielectric(1.5)
            pool.add_sphere(center, 0.2, m, vel)
    return tracer


def penultimate_scene(img_w: int, devices=(0,)) -> Tracer:
    """penultimateScene (rayz.zig:170-239) — dead code in the reference (it targets a removed MemPool API), restated with
    today's calls in its insertion order: diffuse centre sphere, ground, a glass sphere with an air bubble inside it
    (refractive index 1/1.5: hollow glass), and a fully fuzzy metal sphere.  Camera: vfov 20, focus 3.4, defocus 10 degrees."""
    tracer = Tracer(img_w, 20.0, 3.4, 10.0, (-2, 2, 1), (0, 0, -1), (0, 1, 0), devices=devices)
    pool = tracer.pool
    pool.add_sphere((0, 0, -1.2), 0.5, pool.add_diffuse(pool.add_solid((0.1, 0.2, 0.5))))
    pool.add_sphere((0, -100.5, -1), 100, pool.add_diffuse(pool.add_solid((0.8, 0.8, 0.0))))
    pool.add_sphere((-1, 0, -1), 0.5, pool.add_dielectric(1.5))            # left outer
    pool.add_sphere((-1, 0, -1), 0.4, pool.add_dielectric(1.0 / 1.5))      # left inner bubble
    pool.add_sphere((1, 0, -1), 0.5, pool.add_metallic(pool.add_solid((0.8, 0.6, 0.2)), 1.0))
    return tracer
