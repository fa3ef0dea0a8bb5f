"""Time, kernel times and quality of the denoiser (rayz_cuda_denoise), one JSON file.

    python scripts/denoise_probe.py --out OUT_DIR [--runs 7]

With the card's name and power limit read in the same call (randomBouncing seed 42, BVH variant, depth 50):
  * call time: host wall clock around rayz_cuda_denoise (5 iterations, both host outputs copied out; the call ends in a
    device synchronise), median of --runs calls after two warm-up calls, at config 2 (1200 x 675) and 3840 x 2160;
  * kernel times: torch.profiler CUDA activities of the same calls in a separate pass, per kernel name, against the byte floor
    of the algorithm's DRAM traffic (per pixel and level: the (rgb, v) buffer read and written, the normal + depth and
    gradient read, 56 B; prepare and finish read and write their buffers once) at 7.7 TB/s;
  * quality on config 2: PSNR of the linear frame against a 4096-spp frame of independent samples (offset 4096) for 16 and
    64 spp, noisy and denoised (guides of the render's own samples, and of 64 samples), the uniform spp whose noisy PSNR
    reaches the denoised 16-spp PSNR (own-sample guides), and the time of both (render + guides + denoise, and the plain
    render).
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
    ap.add_argument("--runs", type=int, default=7)
    a = ap.parse_args()
    sys.path.insert(0, ROOT)
    import numpy as np
    import torch

    import rayz_b200
    from rayz_b200 import Backend

    res = {"card": card()}
    scene = rayz_b200.random_bouncing(1200, seed=42).pool.arrays()
    b = Backend((0,))
    b.upload_scene(scene)

    def cam(w):
        h = int(w / rayz_b200.ASPECT_RATIO)
        return rayz_b200.Camera.init(20.0, 10.0, 0.6, (13, 2, 3), (0, 0, 0), (0, 1, 0), h, w).rz, h

    def p(w, h, spp, **kw):
        return Backend.params(w, h, spp, 50, seed=1, variant="bvh", **kw)

    def timed(fn):
        t0 = time.perf_counter()
        fn()
        return (time.perf_counter() - t0) * 1e3

    # ---- call time and kernel times
    sizes = {"config2_1200x675": 1200, "3840x2160": 3840}
    res["call_ms"], res["kernels"] = {}, {}
    for name, w in sizes.items():
        c, h = cam(w)
        b.render(c, p(w, h, 16, moments=True))
        b.guides(c, p(w, h, 16))
        for _ in range(2):
            b.denoise()
        t = sorted(timed(b.denoise) for _ in range(a.runs))
        res["call_ms"][name] = {"runs": t, "median": t[len(t) // 2], "pixels": w * h}
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(a.runs):
                b.denoise()
            torch.cuda.synchronize()
        ks = {}
        for e in prof.key_averages():
            if "denoise" in e.key or "atrous" in e.key or "resolve" in e.key:
                ks[e.key] = {"count": e.count, "total_us": e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total}
        px = w * h
        floor = {"prepare": px * (16 + 4 + 16 + 16 + 16 + 8) / 7.7e12 * 1e6, "atrous_level": px * 56 / 7.7e12 * 1e6,
                 "finish": px * (16 + 16 + 16 + 3) / 7.7e12 * 1e6}
        res["kernels"][name] = {"per_kernel": ks, "byte_floor_us": floor}
        print(name, res["call_ms"][name]["median"], ks, floor, flush=True)

    # ---- quality on config 2
    c, h = cam(1200)
    ref, _, _ = b.render(c, p(1200, h, 4096, sample_offset=4096))
    ref = ref[..., :3].astype(np.float64)
    psnr = lambda x: float(10 * np.log10(1.0 / ((np.clip(x[..., :3], 0, None) - ref) ** 2).mean()))
    q = {}
    for spp in (16, 64):
        noisy, _, _ = b.render(c, p(1200, h, spp, moments=True))
        b.guides(c, p(1200, h, spp))
        den, _ = b.denoise()
        b.guides(c, p(1200, h, 64))
        den64, _ = b.denoise()
        q[spp] = {"noisy_psnr": psnr(noisy), "denoised_psnr": psnr(den), "denoised_psnr_64spp_guides": psnr(den64)}
    target = q[16]["denoised_psnr"]
    curve = {}
    for spp in (16, 32, 64, 128, 256, 512, 1024, 2048):
        lin, _, _ = b.render(c, p(1200, h, spp))
        curve[spp] = psnr(lin)
    reach = next((s for s, v in curve.items() if v >= target), None)
    c16 = p(1200, h, 16, moments=True)
    for _ in range(2):
        b.render(c, c16); b.guides(c, p(1200, h, 16)); b.denoise()
    t_den = sorted(timed(lambda: (b.render(c, c16), b.guides(c, p(1200, h, 16)), b.denoise())) for _ in range(a.runs))
    t_plain = None
    if reach:
        pr = p(1200, h, reach)
        b.render(c, pr)
        t_plain = sorted(timed(lambda: b.render(c, pr)) for _ in range(a.runs))
    res["quality_config2"] = {"psnr": q, "noisy_psnr_by_spp": curve, "uniform_spp_reaching_denoised_16spp": reach,
                              "render16_guides16_denoise_ms": t_den[len(t_den) // 2],
                              "plain_render_ms_at_that_spp": t_plain[len(t_plain) // 2] if t_plain else None}
    print(json.dumps(res["quality_config2"]), flush=True)
    b.close()
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "denoise_probe.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
