"""Cost of adaptive sampling on config 2 (1200x675, depth 50, randomBouncing seed 42, start 16 spp, max 4096 spp), one JSON file.

    python scripts/adaptive_probe.py --out OUT_DIR [--runs 3]

For per-pixel targets of 2/255 and 1/255 it reports, with the card's name and power limit read in the same call:
  * adaptive  : rayz_cuda_render_to_noise with RZ_RENDER_ADAPTIVE: wall time, total paths, mean and max spp, rounds, the
                pixels each round listed (and the share of the last work unit's 32 lanes they fill), rms and max error;
  * max_uniform : uniform doubling batches (RZ_RENDER_ACCUMULATE, render + rayz_cuda_noise per batch here) until the frame's
                MAX error reaches the same target, or max_spp: what a caller needs without adaptive sampling for the same bound;
  * rms_uniform : rayz_cuda_render_to_noise (uniform) with the same value as an RMS target.
The arms alternate within each run, after one warm-up call of each.  Times are host wall clock around calls that end in a
device synchronise; AUTO variant, device-resident except the final copy of render_to_noise's RGB8 frame.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
W, SPP0, MAX_SPP, DEPTH = 1200, 16, 4096, 50


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

    t = rayz_b200.random_bouncing(W, seed=42)
    be = Backend((0,))
    be.upload_scene(t.pool.arrays())
    cam, h = t.camera.rz, t.img.h
    npx = W * h
    p0 = Backend.params(W, h, SPP0, DEPTH, seed=1)

    def timed(fn):
        t0 = time.perf_counter()
        r = fn()
        return (time.perf_counter() - t0) * 1e3, r

    def adaptive(target):
        ms, r = timed(lambda: be.render_to_noise(cam, p0, target, MAX_SPP, want_linear=False, adaptive=True))
        counts = be.pixel_samples().astype(np.int64)
        steps = [SPP0]
        while steps[-1] < int(counts.max()):
            steps.append(steps[-1] + min(steps[-1], MAX_SPP - steps[-1]))
        listed = [int((counts >= s).sum()) for s in steps[1:]]   # the pixels each round after the first traced
        return {"ms": ms, "paths": r[2], "mean_spp": float(counts.mean()), "max_spp": int(counts.max()), "rounds": len(steps),
                "listed_per_round": listed, "last_unit_fill": [(n % 32 or 32) / 32 for n in listed],
                "rms_err": r[3]["rms_err"], "max_err": r[3]["max_err"], "pixels_above": r[3]["n_above"]}

    def max_uniform(target):
        def run():
            done, k = 0, SPP0
            while True:
                be.render_device(cam, Backend.params(W, h, k, DEPTH, seed=1, sample_offset=done, moments=True, accumulate=done > 0), sync=True)
                done += k
                _, nz = be.noise(target)
                if nz["max_err"] <= target or done >= MAX_SPP:
                    return done, nz
                k = min(done, MAX_SPP - done)
        ms, (done, nz) = timed(run)
        return {"ms": ms, "paths": npx * done, "spp": done, "rms_err": nz["rms_err"], "max_err": nz["max_err"], "pixels_above": nz["n_above"]}

    def rms_uniform(target):
        ms, r = timed(lambda: be.render_to_noise(cam, p0, target, MAX_SPP, want_linear=False))
        return {"ms": ms, "paths": r[2], "spp": r[3]["samples"], "rms_err": r[3]["rms_err"], "max_err": r[3]["max_err"],
                "pixels_above": r[3]["n_above"]}

    arms = {"adaptive": adaptive, "max_uniform": max_uniform, "rms_uniform": rms_uniform}
    targets = {"2/255": 2 / 255, "1/255": 1 / 255}
    res = {"card": card(), "workload": f"config 2: randomBouncing seed 42, {W}x{h}, depth {DEPTH}, start {SPP0} spp, max {MAX_SPP} spp, AUTO",
           "runs": a.runs}
    for name, target in targets.items():
        for fn in arms.values():   # warm-up
            fn(target)
        series = {k: [] for k in arms}
        for _ in range(a.runs):    # alternated: every arm once per run
            for k, fn in arms.items():
                series[k].append(fn(target))
        out = {}
        for k, v in series.items():
            ms = sorted(x["ms"] for x in v)
            out[k] = {**{f: v[-1][f] for f in v[-1] if f != "ms"}, "ms": [x["ms"] for x in v], "ms_median": ms[len(ms) // 2]}
        res[name] = out
    res["card_after"] = card()
    be.close()
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "adaptive_probe.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
