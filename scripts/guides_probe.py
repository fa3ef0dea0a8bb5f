"""Time and cost of the guide buffers (rayz_cuda_render_guides), one JSON file.

    python scripts/guides_probe.py --out OUT_DIR [--runs 3]

With the card's name and power limit read in the same call, it reports host wall-clock times of calls that end in a device
synchronise (the guide call includes the copy of both 32-byte-per-pixel buffers to host memory):
  * config 2 (1200x675, randomBouncing seed 42, AUTO variant, depth 50): the guides at 16, 64 and 500 spp, against the
    500-spp render (rayz_cuda_render, linear + RGB8 copied out), alternated within each run after one warm-up call of each;
  * config 4 (99,856 spheres, grid [-158, 158), device LBVH, 1920x1080): the guides at 16 spp, where the walk dominates.
Per arm: every run's time, the median, and camera samples per second of the median.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else f"nvidia-smi failed: {r.stderr.strip()}"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--runs", type=int, default=3)
    a = ap.parse_args()
    sys.path.insert(0, ROOT)
    import numpy as np

    import rayz_b200
    from rayz_b200 import Backend

    def timed(fn):
        t0 = time.perf_counter()
        fn()
        return (time.perf_counter() - t0) * 1e3

    def run_arms(arms, npx):
        res = {name: [] for name, _, _ in arms}
        for _, fn, _ in arms:
            fn()   # warm-up: module load, first allocations
        for _ in range(a.runs):
            for name, fn, _ in arms:
                res[name].append(timed(fn))
        out = {}
        for name, _, spp in arms:
            med = float(np.median(res[name]))
            out[name] = {"ms": res[name], "median_ms": med, "spp": spp, "Msamples_per_s": npx * spp / (med * 1e-3) / 1e6}
        return out

    report = {"card": card(), "runs": a.runs}
    t = rayz_b200.random_bouncing(1200, seed=42)
    be = Backend((0,))
    be.upload_scene(t.pool.arrays())
    cam, w, h = t.camera.rz, t.img.w, t.img.h
    arms = [(f"guides_{s}spp", (lambda s=s: be.guides(cam, Backend.params(w, h, s, 50, seed=1))), s) for s in (16, 64, 500)]
    arms.append(("render_500spp", lambda: be.render(cam, Backend.params(w, h, 500, 50, seed=1)), 500))
    report["config2"] = run_arms(arms, w * h)
    be.close()

    t4 = rayz_b200.random_bouncing(1920, seed=42, grid_lo=-158, grid_hi=158)
    be4 = Backend((0,))
    be4.upload_scene(t4.pool.arrays())
    cam4, w4, h4 = t4.camera.rz, t4.img.w, t4.img.h
    report["config4"] = run_arms([("guides_16spp", lambda: be4.guides(cam4, Backend.params(w4, h4, 16, 50, seed=1)), 16)], w4 * h4)
    be4.close()

    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "guides_probe.json"), "w") as f:
        json.dump(report, f, indent=1)
    print(json.dumps(report))


if __name__ == "__main__":
    main()
