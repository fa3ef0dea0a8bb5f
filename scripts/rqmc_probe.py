"""What the randomised-QMC noise estimate (RZ_RENDER_RQMC) buys and costs, against Philox and plain Sobol, one JSON file.

    python scripts/rqmc_probe.py --out OUT_DIR [--runs 3]

With the card's name and power limit read in the same call (depth 50):
  * calibration at 320 x 180 (config 2 and penultimate_scene, 16 and 64 spp, 4 seeds): the frame mean of the estimate's e^2
    over the measured displayed-value MSE against a 16384-spp Philox reference (two 8192-spp halves; their noise is removed),
    for each sampler (Philox and Sobol read e from the iid formula, RQMC from the pooled replicates);
  * quality at 320 x 180: the excess-MSE ratios RQMC/Philox, Sobol/Philox and RQMC/Sobol at 4, 16 and 64 spp;
  * stopping at 1200 x 675 on both scenes: rayz_cuda_render_to_noise, rms and adaptive, at 2/255 and 1/255 (start 4 spp, cap
    4096): paths, wall time, the estimate and the measured rms displayed error of the returned frame, per sampler;
  * speed: Mpaths/s of a 1200 x 675, 64-spp render with and without the flag over Sobol (AUTO and the BVH variant), alternated;
  * the segment pass's device time (rz_segment_kernel, which computes the gains) (torch.profiler) at 1200 x 675 and 3840 x 2160.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SAMPLERS = {"philox": {}, "sobol": {"sobol": True}, "rqmc": {"sobol": True, "rqmc": True}}


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
    luma = lambda x: 0.2126 * x[..., 0] + 0.7152 * x[..., 1] + 0.0722 * x[..., 2]
    disp = lambda x: np.sqrt(np.maximum(luma(x), 1e-4))

    def setup(name, w):
        t = rayz_b200.random_bouncing(w, seed=42) if name == "config2" else rayz_b200.penultimate_scene(w)
        h = int(w / rayz_b200.ASPECT_RATIO)
        b = Backend((0,))
        b.upload_scene(t.pool.arrays())
        cam = t.camera.rz
        ra, _, _ = b.render(cam, Backend.params(w, h, 8192, 50, seed=1001, variant="bvh"), want_rgb8=False)
        rc, _, _ = b.render(cam, Backend.params(w, h, 8192, 50, seed=1002, variant="bvh"), want_rgb8=False)
        ra, rc = ra[..., :3].astype(np.float64), rc[..., :3].astype(np.float64)
        ref = (ra + rc) / 2
        return dict(b=b, cam=cam, w=w, h=h, ref=ref, ref_var=float(((ra - rc) ** 2).mean()) / 4,
                    ref_disp=float(((disp(ra) - disp(rc)) ** 2).mean()) / 4)

    def disp_mse(S, lin):
        return float(((disp(lin[..., :3].astype(np.float64)) - disp(S["ref"])) ** 2).mean()) - S["ref_disp"]

    # ---- calibration and quality at 320 x 180
    cal, qual = {}, {}
    for name in ("config2", "penultimate"):
        S = setup(name, 320)
        b, cam, w, h = S["b"], S["cam"], S["w"], S["h"]
        for spp in (4, 16, 64):
            ex = {}
            for s, kw in SAMPLERS.items():
                e2, d2, x = [], [], []
                for seed in (31, 32, 33, 34):
                    lin, _, _ = b.render(cam, Backend.params(w, h, spp, 50, seed=seed, variant="bvh", moments=True, **kw), want_rgb8=False)
                    err, _ = b.noise()
                    e2.append(float((err.astype(np.float64) ** 2).mean()))
                    d2.append(disp_mse(S, lin))
                    x.append(float(((lin[..., :3] - S["ref"]) ** 2).mean()) - S["ref_var"])
                if spp in (16, 64):
                    cal[f"{name}_{spp}_{s}"] = float(np.mean(e2) / np.mean(d2))
                ex[s] = float(np.mean(x))
            qual[f"{name}_{spp}"] = {"rqmc/philox": ex["rqmc"] / ex["philox"], "sobol/philox": ex["sobol"] / ex["philox"],
                                     "rqmc/sobol": ex["rqmc"] / ex["sobol"]}
            print(name, spp, qual[f"{name}_{spp}"], {k: v for k, v in cal.items() if k.startswith(f"{name}_{spp}")}, flush=True)
        b.close()
    res["calibration_e2_over_measured"] = cal
    res["excess_mse_ratio"] = qual

    # ---- stopping at 1200 x 675
    stop = {}
    for name in ("config2", "penultimate"):
        S = setup(name, 1200)
        b, cam, w, h = S["b"], S["cam"], S["w"], S["h"]
        for target_steps in (2, 1):
            target = target_steps / 255
            for adaptive in (False, True):
                for s, kw in SAMPLERS.items():
                    p = Backend.params(w, h, 4, 50, seed=61, variant="bvh", **kw)
                    b.render_to_noise(cam, p, target, 4096, adaptive=adaptive)     # warm-up of the same shapes
                    t0 = time.perf_counter()
                    lin, _, paths, nz = b.render_to_noise(cam, p, target, 4096, adaptive=adaptive)
                    dt = time.perf_counter() - t0
                    row = {"paths": paths, "wall_s": dt, "samples": nz["samples"], "rms_estimate": nz["rms_err"], "max_estimate": nz["max_err"],
                           "measured_rms": float(np.sqrt(max(disp_mse(S, lin), 0.0)))}
                    key = f"{name}_{target_steps}/255_{'adaptive' if adaptive else 'rms'}_{s}"
                    stop[key] = row
                    print(key, row, flush=True)
        b.close()
    res["render_to_noise_1200"] = stop

    # ---- speed of the flag over plain Sobol, and the gain kernel's time
    W, H = 1200, 675
    t = rayz_b200.random_bouncing(W, seed=42)
    b = Backend((0,))
    b.upload_scene(t.pool.arrays())
    cam = t.camera.rz

    def timed(p):
        b.render(cam, p, want_linear=False, want_rgb8=False)
        ts = []
        for _ in range(a.runs):
            t0 = time.perf_counter()
            b.render(cam, p, want_linear=False, want_rgb8=False)
            ts.append(time.perf_counter() - t0)
        return float(np.median(ts))

    speed = {}
    for variant in ("auto", "bvh"):
        row = {}
        for rq in (False, True, False, True):
            s = timed(Backend.params(W, H, 64, 50, seed=1, variant=variant, moments=True, sobol=True, rqmc=rq))
            row.setdefault("rqmc" if rq else "sobol_moments", []).append(W * H * 64 / s / 1e6)
        row["cost"] = 1 - np.median(row["rqmc"]) / np.median(row["sobol_moments"])
        speed[variant] = row
        print("speed", variant, row, flush=True)
    res["mpaths_per_s_64spp_1200"] = speed

    import torch
    from torch.profiler import ProfilerActivity, profile
    gk = {}
    for w in (1200, 3840):
        h = int(w / rayz_b200.ASPECT_RATIO)
        cw = rayz_b200.random_bouncing(w, seed=42).camera.rz
        b.render(cw, Backend.params(w, h, 4, 50, seed=1, variant="bvh", moments=True, sobol=True, rqmc=True), want_rgb8=False)
        b.noise()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(20):
                b.noise()
        ev = [e for e in prof.events() if "rz_segment_kernel" in e.name]
        gk[f"{w}x{h}"] = {"calls": len(ev), "mean_us": float(np.mean([e.device_time for e in ev])) if ev else None}
        print("gain kernel", w, gk[f"{w}x{h}"], flush=True)
    res["gain_kernel"] = gk
    b.close()

    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "rqmc_probe.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
