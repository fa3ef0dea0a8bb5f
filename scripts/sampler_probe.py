"""Cost and quality of the low-discrepancy sampler (RZ_RENDER_SOBOL) against the default Philox sampler, one JSON file.

    python scripts/sampler_probe.py --out OUT_DIR [--runs 3]

With the card's name and power limit read in the same call (depth 50):
  * speed: Mpaths/s of a 1200 x 675, 64-spp render (51.8 M paths: AUTO runs the BVH kernel), two alternated runs of each
    sampler, each the median of --runs after a warm-up, for randomBouncing seed 42 under AUTO and the BVH variant, its
    glass-heavy version (config 5) and a 2,500-sphere randomBouncing under the BVH variant (a stand-in for config 4's
    many-sphere BVH workload);
  * quality on config 2 at 1200 x 675 against a 16384-spp Philox reference (two independent 8192-spp halves; their noise is
    subtracted): PSNR of the linear frame and render time at 4..256 spp for both samplers under AUTO (from 96 spp, 77.8 M
    paths, AUTO runs the staged K1: those times are its cost), the PSNR of the largest Sobol frame that takes no longer than
    Philox's 64-spp frame (equal time), and the spp Sobol needs to reach Philox's 64-spp PSNR (equal quality, interpolated in
    log spp);
  * denoising: 16-spp render + guides of the render's own samples + rayz_cuda_denoise, with and without the flag.
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

    res = {"card": card()}
    W = 1200
    H = int(W / rayz_b200.ASPECT_RATIO)

    def timed(b, cam, p):
        b.render(cam, p, want_linear=False, want_rgb8=False)
        ts = []
        for _ in range(a.runs):
            t0 = time.perf_counter()
            b.render(cam, p, want_linear=False, want_rgb8=False)
            ts.append(time.perf_counter() - t0)
        return float(np.median(ts))

    speed = {}
    workloads = [("config2_auto", dict(), "auto"), ("config2_bvh", dict(), "bvh"), ("config5_glass_auto", dict(glass_heavy=True), "auto"),
                 ("spheres2500_bvh", dict(grid_lo=-25, grid_hi=25), "bvh")]
    for name, kw, variant in workloads:
        t = rayz_b200.random_bouncing(W, seed=42, **kw)
        b = Backend((0,))
        b.upload_scene(t.pool.arrays())
        row = {}
        for sobol in (False, True, False, True):
            s = timed(b, t.camera.rz, Backend.params(W, H, 64, 50, seed=1, variant=variant, sobol=sobol))
            row.setdefault("sobol" if sobol else "philox", []).append(W * H * 64 / s / 1e6)
        row["variant_ran"] = b.timing()["variant"]
        row["cost"] = 1 - np.median(row["sobol"]) / np.median(row["philox"])
        speed[name] = row
        b.close()
        print(name, row, flush=True)
    res["mpaths_per_s"] = speed

    t = rayz_b200.random_bouncing(W, seed=42)
    b = Backend((0,))
    b.upload_scene(t.pool.arrays())
    cam = t.camera.rz
    ra, _, _ = b.render(cam, Backend.params(W, H, 8192, 50, seed=1001, variant="auto"), want_rgb8=False)
    rc, _, _ = b.render(cam, Backend.params(W, H, 8192, 50, seed=1002, variant="auto"), want_rgb8=False)
    ra, rc = ra[..., :3].astype(np.float64), rc[..., :3].astype(np.float64)
    ref, ref_var = (ra + rc) / 2, float(((ra - rc) ** 2).mean()) / 4

    def psnr(x):
        return float(10 * np.log10(1.0 / max(float(((x[..., :3] - ref) ** 2).mean()) - ref_var, 1e-30)))

    quality, times = {}, {}
    spps = [4, 8, 16, 32, 48, 64, 96, 128, 256]
    for sobol in (False, True):
        key = "sobol" if sobol else "philox"
        quality[key], times[key] = {}, {}
        for spp in spps:
            p = Backend.params(W, H, spp, 50, seed=21, variant="auto", sobol=sobol)
            lin, _, _ = b.render(cam, p, want_rgb8=False)
            quality[key][spp] = psnr(lin)
            times[key][spp] = timed(b, cam, p)
    res["psnr_config2"] = quality
    res["time_config2_s"] = times
    target = quality["philox"][64]
    ls, qs = np.log(spps), np.array([quality["sobol"][s] for s in spps])
    res["equal_quality_sobol_spp"] = float(np.exp(np.interp(target, qs, ls))) if qs.min() <= target <= qs.max() else None
    within = [s for s in spps if times["sobol"][s] <= times["philox"][64]]
    res["equal_time_sobol_spp"] = max(within) if within else None
    res["equal_time_sobol_psnr"] = quality["sobol"][max(within)] if within else None
    res["equal_time_philox_psnr"] = target

    den = {}
    for sobol in (False, True):
        p = Backend.params(W, H, 16, 50, seed=21, variant="auto", moments=True, sobol=sobol)
        lin, _, _ = b.render(cam, p, want_rgb8=False)
        b.guides(cam, p)
        dl, _ = b.denoise()
        den["sobol" if sobol else "philox"] = {"noisy_psnr": psnr(lin), "denoised_psnr": psnr(dl)}
    res["denoise_16spp_own_guides"] = den
    b.close()

    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "sampler_probe.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
