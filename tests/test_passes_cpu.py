"""CPU tests of light-path passes (RZ_RENDER_PASSES).

1. The pass rule and the seg word's encoding, compiled as host code by tests/hostsim/passes.cu, against a table: every
   (hits, first kind), walks of mixed kinds, the count masked at max_depth's edge values and the refusal bound.
2. The replay's first-hit kind (tests/passes_replay.py) is consistent with the full replay's hits and ends on the replay scenes.
3. The ctypes mirror, the header, the Zig shim and the public layers carry the flag, the pass constants and the entry point."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

import oracle
from passes_replay import pass_of, replay_first
from rayz_b200 import _abi as abi
from replay_scenes import all_materials, config1

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
DIFFUSE, METALLIC, DIELECTRIC = abi.MAT_DIFFUSE, abi.MAT_METALLIC, abi.MAT_DIELECTRIC


@pytest.fixture(scope="module")
def lib():
    subprocess.run(["bash", os.path.join(HERE, "hostsim", "build_passes.sh")], check=True)
    lib = C.CDLL(os.path.join(HERE, "_build", "libhostpass.so"))
    for name in ("hostpass_of", "hostpass_after_hit"):
        getattr(lib, name).argtypes, getattr(lib, name).restype = [C.c_uint32, C.c_uint32], C.c_uint32
    for name in ("hostpass_hits", "hostpass_first_kind"):
        getattr(lib, name).argtypes, getattr(lib, name).restype = [C.c_uint32], C.c_uint32
    lib.hostpass_count.restype = lib.hostpass_max_depth.restype = C.c_uint32
    lib.hostpass_walk.argtypes, lib.hostpass_walk.restype = [C.c_void_p, C.c_uint32], C.c_uint32
    return lib


# the header's table: (hits, first kind) -> pass
TABLE = {(0, None): 0, (1, DIFFUSE): 1, (2, DIFFUSE): 2, (1, METALLIC): 3, (2, METALLIC): 4, (1, DIELECTRIC): 5, (2, DIELECTRIC): 6}


def test_pass_rule_matches_the_table(lib):
    assert lib.hostpass_count() == abi.PASS_COUNT == 7
    for kind in (None, DIFFUSE, METALLIC, DIELECTRIC):
        for hits in (0, 1, 2, 3, 7, 50, 1000, (1 << 29) - 1):
            want = TABLE[(0, None)] if hits == 0 else TABLE[(min(hits, 2), kind)] if kind is not None else None
            if want is None:
                continue
            got = lib.hostpass_of(hits, 0 if kind is None else kind)
            assert got == want == int(pass_of(hits, -1 if kind is None else kind)), (hits, kind, got, want)
    assert [lib.hostpass_of(0, k) for k in range(3)] == [0, 0, 0]   # a miss ignores the kind


def test_walks_take_the_first_hits_kind(lib):
    rng = np.random.default_rng(3)
    walks = [[], [DIFFUSE], [METALLIC], [DIELECTRIC], [DIELECTRIC, DIELECTRIC, DIFFUSE], [METALLIC, DIFFUSE], [DIFFUSE, METALLIC, DIELECTRIC]]
    walks += [list(rng.integers(0, 3, int(rng.integers(1, 60)))) for _ in range(200)]
    for w in walks:
        a = np.array(w, dtype=np.uint32)
        want = 0 if not w else TABLE[(min(len(w), 2), int(w[0]))]
        assert lib.hostpass_walk(a.ctypes.data, len(w)) == want, w


def test_seg_word_encoding_and_masking(lib):
    top = lib.hostpass_max_depth()
    assert top == (1 << 29) - 1   # the refusal bound: max_depth above it is refused (the count would reach bit 29)
    for kind in (DIFFUSE, METALLIC, DIELECTRIC):
        s = lib.hostpass_after_hit(0, kind)                        # the first hit records the kind
        assert lib.hostpass_hits(s) == 1 and lib.hostpass_first_kind(s) == kind
        for other in (DIFFUSE, METALLIC, DIELECTRIC):              # later hits keep it
            t = lib.hostpass_after_hit(s, other)
            assert lib.hostpass_hits(t) == 2 and lib.hostpass_first_kind(t) == kind
        # the count at the edge of the largest accepted max_depth: it never spills into the kind bits
        edge = (kind << 29) | (top - 1)
        e = lib.hostpass_after_hit(edge, DIFFUSE)
        assert lib.hostpass_hits(e) == top and lib.hostpass_first_kind(e) == kind and e >> 31 == 0
        assert lib.hostpass_of(lib.hostpass_hits(e), lib.hostpass_first_kind(e)) == 2 + 2 * kind
        # bit 31 (the wavefront's dead-on-arrival marker) is neither a hit nor a kind
        assert lib.hostpass_hits((1 << 31) | (kind << 29) | 5) == 5 and lib.hostpass_first_kind((1 << 31) | (kind << 29) | 5) == kind
    # without the flag's instances seg is the plain count: a count below the bound has no kind bits set
    assert lib.hostpass_first_kind(top) == 0 and lib.hostpass_hits(top) == top


@pytest.mark.parametrize("name", ["config1", "glass", "all_outside", "all_in_glass"])
def test_replay_first_hit_is_consistent(name):
    if name.startswith("all"):
        arrays, cams, w, h = all_materials()
        cam = cams["outside" if name == "all_outside" else "in_glass"]
        w, h = 101, 57
        cam = oracle.camera(*((30.0, 3.4, 2.0, (-2, 2, 1)) if name == "all_outside" else (70.0, 2.0, 0.0, (0.5, 0.6, 0.8))),
                            (0, 0, -1), (0, 1, 0), h, w)
    else:
        w, h = 96, 54
        arrays, cam = config1(w, h, glass_heavy=name == "glass")
    sc = oracle.Scene.from_arrays(arrays)
    for sampler in ("philox", "sobol"):
        full = sc.replay(cam, w, h, 0, 2, 50, seed=11, sampler=sampler)
        first, one = replay_first(sc, cam, w, h, 0, 2, seed=11, sampler=sampler)
        hits = full["hits"].sum(axis=-1)
        rob = full["robust"]
        # a camera ray that missed has no hits and ends in the sky; one that hit has a hit of its first kind
        assert ((first < 0) == (hits == 0))[rob].all()
        assert (full["end"][rob & (first < 0)] == oracle.END_SKY).all()
        idx = np.clip(first, 0, 2)[..., None]
        assert (np.take_along_axis(full["hits"], idx, axis=-1)[..., 0] >= 1)[rob & (first >= 0)].all()
        # a path with hits of one kind only started with it
        single = (np.count_nonzero(full["hits"], axis=-1) == 1) & rob
        assert (first[single] == full["hits"].argmax(axis=-1)[single]).all()
        # the depth-1 replay stops at that first hit (or reaches the sky): at most one hit, one segment
        assert (one["segs"] <= 1).all() and (one["hits"].sum(axis=-1) <= 1).all()
        # the scenes exercise several passes each, transmission in all of them
        sky = rob & (full["end"] == oracle.END_SKY)
        seen = set(np.unique(pass_of(hits[sky], first[sky])).tolist())
        assert len(seen) >= 3 and {5, 6} <= seen, (name, sampler, seen)


def test_flag_constants_and_entry_point_in_every_layer():
    hdr = open(os.path.join(ROOT, "include", "rayz_cuda.h")).read()
    assert int(re.search(r"#define RZ_RENDER_PASSES (0x[0-9a-f]+)u", hdr).group(1), 16) == abi.RENDER_PASSES == 0x80
    names = re.findall(r"RZ_PASS_([A-Z_]+) = (\d+)", hdr)
    enum = {n.lower(): int(v) for n, v in names if n != "COUNT"}
    assert [enum[n] for n in abi.PASS_NAMES] == list(range(7)) and dict(names)["COUNT"] == "7"
    assert "int rayz_cuda_passes(RzContext *ctx, float *out_passes);" in hdr
    assert "rayz_cuda_passes" in abi.SYMBOLS
    zig = open(os.path.join(ROOT, "zig", "cuda_backend.zig")).read()
    assert "pub const RZ_RENDER_PASSES: u32 = 0x80;" in zig and "pub extern fn rayz_cuda_passes(" in zig
    for n in abi.PASS_NAMES:
        assert f"pub const RZ_PASS_{n.upper()}: u32 = {abi.PASS_NAMES.index(n)};" in zig
    cpp = open(os.path.join(ROOT, "host", "rayz_host.cpp")).read()
    assert '"--passes"' in cpp and all(f'"{n}"' in cpp for n in abi.PASS_NAMES)
    from rayz_b200 import Backend
    assert Backend.params(8, 8, 1, passes=True).flags == abi.RENDER_PASSES
    assert Backend.params(8, 8, 1).flags & abi.RENDER_PASSES == 0
    lib = abi.load()   # the library exports the entry point (load() binds every declared symbol)
    assert hasattr(lib, "rayz_cuda_passes")
