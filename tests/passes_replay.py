"""The light-path pass of every replayed path (include/rayz_cuda.h "Light-path passes"), shared by test_passes_cpu.py and
test_passes_gpu.py.

The oracle's replay (oracle Scene.replay) reports a path's hits per material kind; the pass also needs the kind of its FIRST
hit.  Every uniform is a pure function of (seed, pixel, sample, bounce), so a replay of the same frame with depth 1 traces the
same camera rays to the same first hits and stops there: its one counted hit is the first hit of the full replay's path."""
import numpy as np

PASS_ENVIRONMENT = 0


def pass_of(hits, first):
    """rz_pass_of in numpy: hits = scattering hits before the sky, first = RZ_MAT_* of the first hit (ignored when hits = 0)."""
    hits, first = np.asarray(hits), np.asarray(first)
    return np.where(hits == 0, PASS_ENVIRONMENT, 1 + 2 * np.maximum(first, 0) + (hits >= 2))


def replay_first(scene, cam, w, h, sample_offset, spp, seed, t_min=0.0, sampler="philox"):
    """The material kind of each path's first hit, -1 for a camera ray that missed: [h, w, spp] int, from a depth-1 replay."""
    one = scene.replay(cam, w, h, sample_offset, spp, 1, seed=seed, t_min=t_min, sampler=sampler)
    hit = one["hits"].sum(axis=-1) > 0
    return np.where(hit, one["hits"].argmax(axis=-1), -1), one
