"""Cost of the light-path passes (RZ_RENDER_PASSES), one JSON file.

    python scripts/passes_probe.py --out OUT_DIR [--runs 5]

With the card's name and power limit read in the same call, it times config 2 (1200x675, randomBouncing seed 42, 500 spp,
depth 50, render seed 1) with the flag off and on, for the AUTO variant (staged K1 with the BVH tail) and the BVH variant
(staged K3), Philox and Sobol: device kernel time (RzTiming.kernel_ms) and host wall time of rayz_cuda_render (linear + RGB8
copied out), arms alternated within each run after one warm-up call of each.  It also times rayz_cuda_passes itself and checks
that the flag changed no pixel and that the passes sum to the frame (largest deviation in f32 ulp).
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
    ap.add_argument("--runs", type=int, default=5)
    a = ap.parse_args()
    sys.path.insert(0, ROOT)
    import numpy as np

    import rayz_b200
    from rayz_b200 import Backend

    t = rayz_b200.random_bouncing(1200, seed=42)
    be = Backend((0,))
    be.upload_scene(t.pool.arrays())
    cam, w, h, spp = t.camera.rz, 1200, 675, 500
    report = {"card": card(), "runs": a.runs, "frame": f"config 2, {w}x{h}, {spp} spp, depth 50", "arms": {}}
    for variant in ("auto", "bvh"):
        for sampler in ("philox", "sobol"):
            arms = {flag: Backend.params(w, h, spp, 50, seed=1, variant=variant, sobol=sampler == "sobol", passes=flag == "on")
                    for flag in ("off", "on")}
            res = {flag: {"kernel_ms": [], "wall_ms": []} for flag in arms}
            outs = {}
            for flag, p in arms.items():   # warm-up, and the outputs to compare
                outs[flag] = be.render(cam, p)[0]
            passes = be.passes()
            for _ in range(a.runs):
                for flag, p in arms.items():
                    t0 = time.perf_counter()
                    be.render(cam, p)
                    res[flag]["wall_ms"].append((time.perf_counter() - t0) * 1e3)
                    res[flag]["kernel_ms"].append(be.timing()["kernel_ms"])
            t0 = time.perf_counter()
            be.passes()
            passes_ms = (time.perf_counter() - t0) * 1e3
            lin = outs["on"]
            s = passes[..., :3].astype(np.float64).sum(axis=0)
            ulp = np.spacing(np.abs(lin[..., :3])).astype(np.float64)
            med = {f: {k: float(np.median(v)) for k, v in r.items()} for f, r in res.items()}
            report["arms"][f"{variant}/{sampler}"] = {
                "runs": res, "median": med,
                "kernel_cost_pct": 100.0 * (med["on"]["kernel_ms"] / med["off"]["kernel_ms"] - 1.0),
                "wall_cost_pct": 100.0 * (med["on"]["wall_ms"] / med["off"]["wall_ms"] - 1.0),
                "image_identical": bool(np.array_equal(outs["off"].view(np.uint32), outs["on"].view(np.uint32))),
                "sum_max_ulp": float(np.max(np.abs(s - lin[..., :3]) / np.maximum(ulp, 1e-45))),
                "rayz_cuda_passes_ms": passes_ms,
                "Mpaths_per_s": {f: w * h * spp / (med[f]["kernel_ms"] * 1e-3) / 1e6 for f in med},
            }
            print(variant, sampler, json.dumps({k: v for k, v in report["arms"][f"{variant}/{sampler}"].items() if k != "runs"}), flush=True)
    be.close()
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "passes_probe.json"), "w") as f:
        json.dump(report, f, indent=1)


if __name__ == "__main__":
    main()
