"""CPU tests of the ID mattes (include/rayz_cuda.h "ID mattes"): the rank key compiled as host code (tests/hostsim/mattes.cu)
against numpy's order, the declarations in every layer, and the replay's first-hit ids the GPU tests compare against."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

import oracle
from rayz_b200 import _abi as abi
import mattes_replay
import passes_replay
import replay_scenes

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = open(os.path.join(ROOT, "include", "rayz_cuda.h")).read()
ZIG = open(os.path.join(ROOT, "zig", "cuda_backend.zig")).read()


@pytest.fixture(scope="module")
def lib():
    subprocess.run(["bash", os.path.join(ROOT, "tests", "hostsim", "build_mattes.sh")], check=True)
    L = C.CDLL(os.path.join(ROOT, "tests", "_build", "libhostmatte.so"))
    L.hostmatte_miss.restype = L.hostmatte_empty.restype = C.c_int32
    L.hostmatte_max_ranks.restype = L.hostmatte_max_spp.restype = C.c_uint32
    L.hostmatte_keys.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p]
    L.hostmatte_decode.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p]
    return L


def keys_of(lib, count, ids):
    count, ids = np.ascontiguousarray(count, np.uint32), np.ascontiguousarray(ids, np.int32)
    keys = np.empty(len(count), np.uint64)
    lib.hostmatte_keys(count.ctypes.data, ids.ctypes.data, len(count), keys.ctypes.data)
    return keys


# ------------------------------------------------------------------------------- 1. the rank key
def test_key_order_is_count_descending_then_id_ascending(lib):
    rng = np.random.default_rng(7)
    big = np.iinfo(np.int32).max
    for trial in range(200):
        n = int(rng.integers(1, 300))
        ids = rng.choice(np.concatenate([[-1, 0, big, big - 1], rng.integers(0, 2 ** 31 - 1, 1000)]), n, replace=False)
        count = rng.integers(0, 4 if trial % 2 else 1025, n)   # few distinct counts: many ties
        if trial % 3 == 0:
            count[:2] = (0, 1024)
        keys = keys_of(lib, count, ids)
        assert len(np.unique(keys)) == n   # distinct ids give distinct keys
        want = np.lexsort((ids, -count.astype(np.int64)))
        assert np.array_equal(np.argsort(keys, kind="stable"), want)
        got_c, got_i = np.empty(n, np.uint32), np.empty(n, np.int32)
        lib.hostmatte_decode(keys.ctypes.data, n, got_c.ctypes.data, got_i.ctypes.data)
        assert np.array_equal(got_c, count) and np.array_equal(got_i, ids)


def test_empty_and_miss_ids_decode(lib):
    for cnt, i in ((0, -2), (1024, -1), (5, 0), (1, np.iinfo(np.int32).max), (1024, np.iinfo(np.int32).min)):
        k = keys_of(lib, [cnt], [i])
        c, d = np.empty(1, np.uint32), np.empty(1, np.int32)
        lib.hostmatte_decode(k.ctypes.data, 1, c.ctypes.data, d.ctypes.data)
        assert (int(c[0]), int(d[0])) == (cnt, i)


# ------------------------------------------------------------------------------- 2. declarations in every layer
def test_constants_match_header_abi_zig_and_device(lib):
    for name, py in (("RZ_MATTE_MISS", abi.MATTE_MISS), ("RZ_MATTE_EMPTY", abi.MATTE_EMPTY),
                     ("RZ_MATTE_MAX_RANKS", abi.MATTE_MAX_RANKS), ("RZ_MATTE_MAX_SPP", abi.MATTE_MAX_SPP)):
        m = re.search(r"#define %s\s+\(?(-?\d+)u?\)?" % name, HEADER)
        assert m and int(m.group(1)) == py, name
        z = re.search(r"pub const %s: [iu]32 = (-?\d+);" % name, ZIG)
        assert z and int(z.group(1)) == py, name
    assert (lib.hostmatte_miss(), lib.hostmatte_empty(), lib.hostmatte_max_ranks(), lib.hostmatte_max_spp()) == \
        (abi.MATTE_MISS, abi.MATTE_EMPTY, abi.MATTE_MAX_RANKS, abi.MATTE_MAX_SPP)


def test_signature_matches_header_abi_and_zig():
    m = re.search(r"int rayz_cuda_render_mattes\(RzContext \*ctx, const RzCamera \*cam, const RzRenderParams \*p, uint32_t ranks,\s*"
                  r"int32_t \*out_ids, float \*out_coverage\);", HEADER)
    assert m
    res, args = abi.SYMBOLS["rayz_cuda_render_mattes"]
    assert res is C.c_int and len(args) == 6 and args[3] is C.c_uint32
    assert "pub extern fn rayz_cuda_render_mattes(ctx: *RzContext, cam: *const RzCamera, params: *const RzRenderParams, " \
           "ranks: u32, out_ids: ?[*]i32, out_coverage: ?[*]f32) c_int;" in ZIG


# ------------------------------------------------------------------------------- 3. the replay's first hits
@pytest.mark.parametrize("sampler", ["philox", "sobol"])
@pytest.mark.parametrize("which", ["config1", "outside", "in_glass"])
def test_replay_first_agrees_with_the_replay(which, sampler):
    """first = -1 exactly where the depth-1 replay counts no hit; the material kind of sphere `first` is the replay's kind of
    the first hit (tests/passes_replay.py); and a full-depth replay proves the same samples' first hits.  Checked on the
    proven samples, where an f64 restatement must agree; they must be nearly all."""
    if which == "config1":
        arrays, cam = replay_scenes.config1(24, 14)
        w, h, t_min = 24, 14, 0.0
    else:
        arrays, cams, w, h = replay_scenes.all_materials()
        cam, t_min = cams[which], (1e-3 if which == "in_glass" else 0.0)
    sc = oracle.Scene.from_arrays(arrays)
    spp, seed = (6 if which == "config1" else 2), 11
    first, proven, one = mattes_replay.replay_first(sc, arrays, cam, w, h, 0, spp, seed, t_min, sampler)
    assert proven.mean() >= 0.95, proven.mean()
    miss = one["hits"].sum(axis=-1) == 0
    assert np.array_equal((first == -1)[proven], miss[proven])
    kind_ref, _ = passes_replay.replay_first(sc, cam, w, h, 0, spp, seed, t_min, sampler)
    kind = np.where(first >= 0, arrays["mat_kind"][arrays["sphere_material"][np.maximum(first, 0)]].astype(np.int64), -1)
    assert np.array_equal(kind[proven], kind_ref[proven])
    full = sc.replay(cam, w, h, 0, spp, 50, seed=seed, t_min=t_min, sampler=sampler)
    full_proven = (full["reason"] == 0) | (full["fseg"] >= 1)
    assert (full_proven | ~proven).all()   # the depth-1 rule is the stricter one
    assert np.array_equal(((full["hits"].sum(axis=-1) == 0) & (full["end"] == oracle.END_SKY))[proven], (first == -1)[proven])
    assert len(np.unique(first[first >= 0])) >= 2   # not vacuous (all_materials shows no sky; in_glass sees two spheres)


def test_ranked_histogram_helper():
    first = np.array([[[3, -1, 3, 0, 2, 2, 2, 3]]])
    hist = mattes_replay.histograms(first, 5)
    assert hist[0, 0].tolist() == [1, 1, 0, 3, 3, 0]
    ids, cnt = mattes_replay.ranked(hist, 6)
    assert ids[0, 0].tolist() == [2, 3, -1, 0, -2, -2] and cnt[0, 0].tolist() == [3, 3, 1, 1, 0, 0]
