"""ctypes declarations of include/rayz_cuda.h and the loader of librayz_cuda.so.

The library is the product; there is no fallback.  `load()` raises if the .so is missing or a
declared symbol is absent, and every compute entry point fails with RZ_ERR_CUDA without a GPU.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(HERE, "lib", "librayz_cuda.so")

RZ_OK = 0
ERRORS = {-1: "RZ_ERR_INVALID_ARG", -2: "RZ_ERR_CUDA", -3: "RZ_ERR_NCCL", -4: "RZ_ERR_OOM", -5: "RZ_ERR_UNSUPPORTED",
          -6: "RZ_ERR_NO_SCENE", -7: "RZ_ERR_INTERNAL"}
MAT_DIFFUSE, MAT_METALLIC, MAT_DIELECTRIC = 0, 1, 2
TEX_CHECKER, TEX_SOLID = 0, 1
DIFFUSE_UNIT_SPHERE, DIFFUSE_UNIT_SPHERE_SURFACE, DIFFUSE_HEMISPHERE = 0, 1, 2
VARIANT_AUTO, VARIANT_MEGA, VARIANT_WAVEFRONT, VARIANT_BVH = 0, 1, 2, 3
VARIANTS = {"auto": 0, "mega": 1, "wavefront": 2, "bvh": 3, "mega_single": 4}
RENDER_SERIAL_PASSES, RENDER_MOMENTS, RENDER_ACCUMULATE, RENDER_ADAPTIVE, RENDER_SOBOL, RENDER_RQMC = 1, 2, 4, 8, 0x10, 0x20   # RzRenderParams.flags (RZ_RENDER_*)
RENDER_ADAPTIVE_POOLED = 0x40   # with RENDER_ADAPTIVE in render_to_noise: stop each pixel on an error pooled over its row segment
RENDER_PASSES = 0x80            # also sum each sky path's radiance into its light-path pass (rayz_cuda_passes)
# pixel reconstruction filter, a field of RzRenderParams.flags (RZ_RENDER_FILTER): kind in bits 8-9, full width in 1/16 px in
# bits 16-23 (0: the kind's default; else 16..64)
RENDER_FILTER_SHIFT, RENDER_FILTER_MASK, RENDER_FILTER_WIDTH_SHIFT, RENDER_FILTER_WIDTH_MASK = 8, 0x300, 16, 0xFF0000
FILTER_BOX, FILTER_TENT, FILTER_GAUSSIAN, FILTER_BLACKMAN_HARRIS = 0, 1, 2, 3
FILTER_WIDTH_MIN, FILTER_WIDTH_MAX = 16, 64
FILTERS = {"box": FILTER_BOX, "tent": FILTER_TENT, "gaussian": FILTER_GAUSSIAN, "blackman-harris": FILTER_BLACKMAN_HARRIS}


def render_filter(kind: int, width16: int = 0) -> int:
    """RZ_RENDER_FILTER(kind, width16): the flags of a filter."""
    return ((kind << RENDER_FILTER_SHIFT) & RENDER_FILTER_MASK) | ((width16 << RENDER_FILTER_WIDTH_SHIFT) & RENDER_FILTER_WIDTH_MASK)


# RZ_PASS_*: index -> name of the light-path passes rayz_cuda_passes returns, in plane order
PASS_NAMES = ("environment", "diffuse_direct", "diffuse_indirect", "glossy_direct", "glossy_indirect", "transmission_direct",
              "transmission_indirect")
PASS_COUNT = len(PASS_NAMES)
# ID mattes (rayz_cuda_render_mattes): the id of a sample that hit no sphere, of a rank past the pixel's distinct ids, and limits
MATTE_MISS, MATTE_EMPTY, MATTE_MAX_RANKS, MATTE_MAX_SPP = -1, -2, 16, 1024

_dp, _up = C.POINTER(C.c_double), C.POINTER(C.c_uint32)


class RzScene(C.Structure):
    _fields_ = [("n_spheres", C.c_uint32), ("n_materials", C.c_uint32), ("n_textures", C.c_uint32), ("reserved0", C.c_uint32),
                ("sphere_center", _dp), ("sphere_velocity", _dp), ("sphere_radius", _dp), ("sphere_material", _up),
                ("mat_kind", _up), ("mat_fuzz", _dp), ("mat_ior", _dp), ("mat_texture", _up), ("mat_method", _up),
                ("tex_kind", _up), ("tex_color", _dp), ("tex_scale", _dp), ("tex_even", _up), ("tex_odd", _up)]


class RzCamera(C.Structure):
    _fields_ = [("look_from", C.c_double * 3), ("px_du", C.c_double * 3), ("px_dv", C.c_double * 3),
                ("px_origin", C.c_double * 3), ("defocus_u", C.c_double * 3), ("defocus_v", C.c_double * 3),
                ("defocus", C.c_int32), ("reserved0", C.c_int32)]


class RzRenderParams(C.Structure):
    _fields_ = [("width", C.c_uint32), ("height", C.c_uint32), ("spp", C.c_uint32), ("max_depth", C.c_uint32),
                ("seed", C.c_uint64), ("sample_offset", C.c_uint32), ("variant", C.c_uint32), ("t_min", C.c_float),
                ("shard_index", C.c_uint32), ("shard_count", C.c_uint32), ("band_rows", C.c_uint32),
                ("collect_stats", C.c_uint32), ("flags", C.c_uint32)]


class RzConfig(C.Structure):
    _fields_ = [("n_devices", C.c_int32), ("device_ids", C.c_int32 * 8), ("flags", C.c_uint32)]


class RzStats(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("paths", "segments", "sphere_tests", "node_tests", "hits_diffuse",
                                          "hits_metallic", "hits_dielectric", "ended_sky", "ended_absorbed", "ended_depth")]

    def as_dict(self):
        return {n: int(getattr(self, n)) for n, _ in self._fields_}


class RzTiming(C.Structure):
    _fields_ = [("kernel_ms", C.c_float), ("resolve_ms", C.c_float), ("total_ms", C.c_float), ("launches", C.c_uint32),
                ("n_static", C.c_uint32), ("n_moving", C.c_uint32), ("variant", C.c_uint32), ("bvh_build_us", C.c_uint32), ("primary_ms", C.c_float), ("passes", C.c_uint32), ("second_ms", C.c_float), ("sort_ms", C.c_float),
                ("sorted_stages", C.c_uint32), ("queue_entries", C.c_uint32)]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_ if n != "reserved0"}


class RzNoise(C.Structure):
    _fields_ = [("samples", C.c_uint64), ("n_pixels", C.c_uint32), ("n_above", C.c_uint32), ("mean_err", C.c_double),
                ("rms_err", C.c_double), ("max_err", C.c_double)]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


class RzTuning(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("rays_per_thread", C.c_int32), ("chunk", C.c_uint32), ("chunk_primary", C.c_uint32),
                ("queue_log2", C.c_int32), ("second_stages", C.c_int32), ("bvh_stages", C.c_int32), ("tail_brute", C.c_int32),
                ("bvh_staged", C.c_int32), ("cell_bits", C.c_int32), ("bvh_active_min", C.c_int32), ("bvh_descend_min", C.c_int32),
                ("sah_leaf", C.c_int32), ("sah_node_cost", C.c_double), ("unit_entries", C.c_uint32), ("debug_queue_cap", C.c_uint32),
                ("debug_stack_cap", C.c_uint32),
                ("key_sectors", C.c_int32), ("lbvh_leaf", C.c_int32), ("huge_factor", C.c_double)]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


class RzDenoiseParams(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("iterations", C.c_uint32), ("sigma_luminance", C.c_float), ("sigma_normal", C.c_float),
                ("sigma_depth", C.c_float), ("reserved0", C.c_uint32)]


# every symbol include/rayz_cuda.h declares: (restype, argtypes)
SYMBOLS = {
    "rayz_cuda_abi_version": (C.c_uint32, []),
    "rayz_cuda_create": (C.c_int, [C.POINTER(RzConfig), C.POINTER(C.c_void_p)]),
    "rayz_cuda_destroy": (None, [C.c_void_p]),
    "rayz_cuda_set_stream": (C.c_int, [C.c_void_p, C.c_void_p]),
    "rayz_cuda_upload_scene": (C.c_int, [C.c_void_p, C.POINTER(RzScene)]),
    "rayz_cuda_reserve": (C.c_int, [C.c_void_p, C.POINTER(RzRenderParams)]),
    "rayz_cuda_render": (C.c_int, [C.c_void_p, C.POINTER(RzCamera), C.POINTER(RzRenderParams), C.c_void_p, C.c_void_p,
                                   C.POINTER(C.c_uint64)]),
    "rayz_cuda_render_device": (C.c_int, [C.c_void_p, C.POINTER(RzCamera), C.POINTER(RzRenderParams), C.POINTER(C.c_void_p),
                                          C.POINTER(C.c_void_p), C.POINTER(C.c_uint64), C.c_int]),
    "rayz_cuda_noise": (C.c_int, [C.c_void_p, C.c_float, C.c_void_p, C.POINTER(RzNoise)]),
    "rayz_cuda_render_to_noise": (C.c_int, [C.c_void_p, C.POINTER(RzCamera), C.POINTER(RzRenderParams), C.c_float, C.c_uint32,
                                            C.c_void_p, C.c_void_p, C.POINTER(C.c_uint64), C.POINTER(RzNoise)]),
    "rayz_cuda_pixel_samples": (C.c_int, [C.c_void_p, C.c_void_p]),
    "rayz_cuda_passes": (C.c_int, [C.c_void_p, C.c_void_p]),
    "rayz_cuda_render_guides": (C.c_int, [C.c_void_p, C.POINTER(RzCamera), C.POINTER(RzRenderParams), C.c_void_p, C.c_void_p]),
    "rayz_cuda_render_mattes": (C.c_int, [C.c_void_p, C.POINTER(RzCamera), C.POINTER(RzRenderParams), C.c_uint32, C.c_void_p,
                                          C.c_void_p]),
    "rayz_cuda_denoise": (C.c_int, [C.c_void_p, C.POINTER(RzDenoiseParams), C.c_void_p, C.c_void_p]),
    "rayz_cuda_shard_rows": (C.c_uint32, [C.c_uint32] * 4),
    "rayz_cuda_context_rows": (C.c_uint32, [C.c_void_p] + [C.c_uint32] * 4),
    "rayz_cuda_primary_ids": (C.c_int, [C.c_void_p, C.POINTER(RzCamera), C.c_uint32, C.c_uint32, C.c_int, C.c_void_p]),
    "rayz_cuda_stats": (C.c_int, [C.c_void_p, C.POINTER(RzStats)]),
    "rayz_cuda_stage_stats": (C.c_int, [C.c_void_p, C.c_uint32, C.POINTER(RzStats)]),
    "rayz_cuda_timing": (C.c_int, [C.c_void_p, C.POINTER(RzTiming)]),
    "rayz_cuda_fp32_peak": (C.c_int, [C.c_void_p, C.c_uint32, C.POINTER(C.c_double), C.POINTER(C.c_int32)]),
    "rayz_cuda_get_tuning": (C.c_int, [C.c_void_p, C.POINTER(RzTuning)]),
    "rayz_cuda_set_tuning": (C.c_int, [C.c_void_p, C.POINTER(RzTuning)]),
    "rayz_cuda_last_error": (C.c_char_p, []),
}
# test hooks outside the reference-facing header
EXTRA_SYMBOLS = {
    "rayz_cuda_debug_sort_keys": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p]),
}

_lib = None


class BackendError(RuntimeError):
    def __init__(self, code: int, text: str):
        super().__init__(f"{ERRORS.get(code, code)}: {text}")
        self.code = code


def load():
    """dlopen librayz_cuda.so and bind every declared symbol; raises if anything is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO_PATH):
        raise ImportError(f"{SO_PATH} is missing: build it with `python -m rayz_b200.build` "
                          "(rayz_b200 has no CPU fallback)")
    lib = C.CDLL(SO_PATH)
    for table in (SYMBOLS, EXTRA_SYMBOLS):
        for name, (res, args) in table.items():
            fn = getattr(lib, name)  # AttributeError if the export is missing
            fn.restype = res
            fn.argtypes = args
    if lib.rayz_cuda_abi_version() != 3:
        raise ImportError("librayz_cuda.so ABI version mismatch")
    _lib = lib
    return lib


def check(rc: int):
    if rc != RZ_OK:
        raise BackendError(rc, load().rayz_cuda_last_error().decode("utf-8", "replace"))
