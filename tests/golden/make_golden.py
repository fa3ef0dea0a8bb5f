"""Generates the committed golden fixtures from the CPU oracle (run in the build container).

    python tests/golden/make_golden.py [--full]

ids_seed42_400x225.npz      primary-ray closest-hit sphere ids of the default scene (config 1 size)
ids_seed42_1200x675.npz     same at config 2 size
ids_config4_960x540.npz     same for BASELINE config 4's scene (randomBouncing with the grid loops widened to [-158, 158):
                            99,856 spheres) at 960x540, through the reference's BVH (hit.zig:130-161,181-216)
scene_seed42.npz            the flat scene arrays of randomBouncing(seed 42) (RzScene field names)
config2_oracle_500spp.npz   (--full) 1200x675, 500 spp, depth 50 oracle render (row-stream mode,
                            seed 2024) reduced to 4x4 and 16x16 block means + global means
config2_oracle_500spp_pixels.npz
                            (--full) the same render at every PIXEL_STEP-th pixel in row-major order: `idx` (flat
                            pixel index), `rgb` (linear float32) — the per-pixel comparison at full resolution
"""
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import oracle  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
PIXEL_STEP = 49   # 16,531 of 810,000 pixels; coprime to the width, so the sample moves across the columns row by row


def block_means(img, b):
    h, w = img.shape[:2]
    hb, wb = h // b, w // b
    return img[:hb * b, :wb * b].reshape(hb, b, wb, b, 3).mean(axis=(1, 3))


def main():
    sc = oracle.Scene.random_bouncing(42)
    np.savez_compressed(os.path.join(HERE, "scene_seed42.npz"), **sc.arrays())
    for w in (400, 1200):
        cam, h = oracle.default_camera(w)
        ids = sc.primary_ids(cam, w, h, use_bvh=True)
        assert ids.max() < 32767
        np.savez_compressed(os.path.join(HERE, f"ids_seed42_{w}x{h}.npz"), ids=ids.astype(np.int16))
        print(w, h, int((ids >= 0).sum()), "hits")
    big = oracle.Scene.random_bouncing(42, -158, 158)
    assert big.counts()[0] == 99856
    cam, h = oracle.default_camera(960)
    ids = big.primary_ids(cam, 960, h, use_bvh=True)
    np.savez_compressed(os.path.join(HERE, f"ids_config4_960x{h}.npz"), ids=ids.astype(np.int32))
    print("config 4:", 960, h, int((ids >= 0).sum()), "hits, max id", int(ids.max()))
    if "--full" in sys.argv:
        cam, h = oracle.default_camera(1200)
        t = time.time()
        img, st = sc.render(cam, 1200, h, 500, 50, seed=2024, threads=0, row_streams=True, stats=True)
        print("500 spp oracle render:", time.time() - t, "s", st)
        idx = np.arange(0, 1200 * h, PIXEL_STEP, dtype=np.uint32)
        np.savez_compressed(os.path.join(HERE, "config2_oracle_500spp_pixels.npz"), idx=idx,
                            rgb=img.reshape(-1, 3)[idx].astype(np.float32), seed=2024, spp=500)
        np.savez_compressed(os.path.join(HERE, "config2_oracle_500spp.npz"),
                            block4=block_means(img, 4).astype(np.float32), block16=block_means(img, 16).astype(np.float32),
                            mean=img.mean(axis=(0, 1)), stats=np.array([st[k] for k in oracle.STAT_NAMES], dtype=np.uint64),
                            seed=2024, spp=500)


if __name__ == "__main__":
    main()
