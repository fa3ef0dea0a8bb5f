"""Cost and look of the pixel filters (RZ_RENDER_FILTER), one JSON file and one PPM per filter.

    python scripts/filter_probe.py --out OUT_DIR [--runs 5]

With the card's name and power limit read in the same call, it renders config 2 (1200x675, randomBouncing seed 42, 500 spp,
depth 50, render seed 1) on the AUTO variant (the staged K1 with the BVH tail) with the box and with each filter at its
default width and at 4 px, arms alternated within each run after one warm-up call of each:
  * Mpaths/s from the device kernel time (RzTiming.kernel_ms);
  * primary_ms, the camera stage's kernel time, with RZ_RENDER_SERIAL_PASSES (the stages run back to back, so that it is the
    primary kernel's own time);
  * sphere tests per camera segment of the primary kernel (rayz_cuda_stage_stats, stage 0, collect_stats), which is what the
    widened tile cones cost;
and writes each arm's converged frame as OUT_DIR/filter_<name>.ppm, to look at the checker ground at the horizon.
"""
from __future__ import annotations

import argparse
import io
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else f"nvidia-smi failed: {r.stderr.strip()}"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--runs", type=int, default=5)
    ap.add_argument("--width", type=int, default=1200)
    ap.add_argument("--spp", type=int, default=500)
    a = ap.parse_args()
    sys.path.insert(0, ROOT)
    import numpy as np

    import rayz_b200
    from rayz_b200 import Backend

    t = rayz_b200.random_bouncing(a.width, seed=42)
    be = Backend((0,))
    be.upload_scene(t.pool.arrays())
    cam, w, h, spp = t.camera.rz, t.img.w, t.img.h, a.spp
    os.makedirs(a.out, exist_ok=True)
    report = {"card": card(), "runs": a.runs, "frame": f"config 2, {w}x{h}, {spp} spp, depth 50, AUTO", "arms": {}}
    arms = {"box": ("box", None)}
    for kind in ("tent", "gaussian", "blackman-harris"):
        arms[f"{kind}"] = (kind, None)
        arms[f"{kind}_4px"] = (kind, 4.0)
    params = {n: Backend.params(w, h, spp, 50, seed=1, pixel_filter=k, filter_width=fw) for n, (k, fw) in arms.items()}
    serial = {n: Backend.params(w, h, spp, 50, seed=1, pixel_filter=k, filter_width=fw, serial_passes=True)
              for n, (k, fw) in arms.items()}
    res = {n: {"kernel_ms": [], "primary_ms": []} for n in arms}
    for n in arms:   # warm-up, the frames, and the camera stage's counters
        lin, rgb8, _ = be.render(cam, params[n])
        t.img.rgb8 = rgb8
        f = io.StringIO()
        t.img.writePPM(f)
        with open(os.path.join(a.out, f"filter_{n}.ppm"), "w") as fh:
            fh.write(f.getvalue())
        be.render(cam, Backend.params(w, h, spp, 50, seed=1, pixel_filter=arms[n][0], filter_width=arms[n][1], collect_stats=True,
                                      serial_passes=True))
        st = be.stage_stats(0)
        report["arms"][n] = {"filter": arms[n], "camera_segments": st["segments"], "sphere_tests": st["sphere_tests"],
                             "sphere_tests_per_camera_segment": st["sphere_tests"] / max(1, st["segments"]),
                             "mean_linear": float(lin[..., :3].mean())}
        be.render(cam, serial[n])
    for _ in range(a.runs):
        for n in arms:
            be.render(cam, params[n])
            res[n]["kernel_ms"].append(be.timing()["kernel_ms"])
            be.render(cam, serial[n])
            res[n]["primary_ms"].append(be.timing()["primary_ms"])
    for n in arms:
        med = {k: float(np.median(v)) for k, v in res[n].items()}
        report["arms"][n].update({"runs": res[n], "median": med, "Mpaths_per_s": w * h * spp / (med["kernel_ms"] * 1e-3) / 1e6})
        print(n, json.dumps({k: v for k, v in report["arms"][n].items() if k != "runs"}), flush=True)
    be.close()
    with open(os.path.join(a.out, "filter_probe.json"), "w") as f:
        json.dump(report, f, indent=1)
    print(report["card"])


if __name__ == "__main__":
    main()
