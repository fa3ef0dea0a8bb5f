"""Cost of progressive rendering on config 2 (1200x675, 500 spp, depth 50, randomBouncing seed 42), one JSON file per call.

    python scripts/progressive_probe.py --out OUT_DIR [--parent-so PATH] [--runs 3]

Reports, with the card's name and power limit read in the same call:
  * default   : config 2 as bench.py renders it (AUTO, device-resident), this build against the parent build's library
                (--parent-so, a librayz_cuda.so built from the parent commit), alternated run by run;
  * moments   : the same with RZ_RENDER_MOMENTS (the fourth atomic per path that ends in the sky) against without;
  * batches   : 500 spp as doubling RZ_RENDER_ACCUMULATE batches (16, 16, 32, 64, 128, 244) against one 500-spp render;
  * to_noise  : rayz_cuda_render_to_noise from 16 spp at rms targets of 2/255 and 1/255 (max 4096 spp): spp reached, ms.
Each measurement runs in its own process (one library per process), one warm-up render first.  Times are host wall
clock around calls that end in a device synchronise.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
W, SPP, DEPTH = 1200, 500, 50


def worker(mode: str, so: str | None, reps: int):
    sys.path.insert(0, ROOT)
    from rayz_b200 import _abi as abi
    if so:   # a library of another commit: bind only what it exports
        abi.SO_PATH = os.path.abspath(so)
        for name in ("rayz_cuda_noise", "rayz_cuda_render_to_noise"):
            abi.SYMBOLS.pop(name, None)
    import rayz_b200
    from rayz_b200 import Backend
    t = rayz_b200.random_bouncing(W, seed=42)
    be = Backend((0,))
    be.upload_scene(t.pool.arrays())
    cam, h = t.camera.rz, t.img.h

    def timed(fn):
        t0 = time.perf_counter()
        r = fn()
        return (time.perf_counter() - t0) * 1e3, r

    def one_shot(moments):
        return be.render_device(cam, Backend.params(W, h, SPP, DEPTH, seed=1, moments=moments), sync=True)

    def doubling():
        done, k = 0, 16
        while done < SPP:
            be.render_device(cam, Backend.params(W, h, k, DEPTH, seed=1, sample_offset=done, moments=True, accumulate=done > 0), sync=True)
            done += k
            k = min(done, SPP - done)

    out = []
    if mode in ("default", "moments_off", "moments_on"):
        one_shot(mode == "moments_on")
        for _ in range(reps):
            ms, _ = timed(lambda: one_shot(mode == "moments_on"))
            out.append({"ms": ms, "kernel_ms": be.timing()["kernel_ms"], "variant": be.timing()["variant"]})
    elif mode in ("batched", "one_shot_moments"):
        fn = doubling if mode == "batched" else (lambda: one_shot(True))
        fn()
        for _ in range(reps):
            ms, _ = timed(fn)
            out.append({"ms": ms})
    elif mode == "to_noise":
        p = Backend.params(W, h, 16, DEPTH, seed=1)
        be.render_to_noise(cam, p, 2 / 255, 4096, want_linear=False)
        for target in (2 / 255, 1 / 255):
            ms, r = timed(lambda: be.render_to_noise(cam, p, target, 4096, want_linear=False))
            out.append({"target": target, "target_in_8bit_steps": target * 255, "ms": ms, "spp": r[3]["samples"],
                        "rms_err": r[3]["rms_err"], "mean_err": r[3]["mean_err"], "max_err": r[3]["max_err"],
                        "pixels_above": r[3]["n_above"]})
    be.close()
    print(json.dumps(out))


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else f"nvidia-smi failed: {r.stderr.strip()}"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--parent-so", default="")
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--worker", default="")
    ap.add_argument("--so", default="")
    ap.add_argument("--reps", type=int, default=2)
    a = ap.parse_args()
    if a.worker:
        return worker(a.worker, a.so or None, a.reps)

    def run(mode, so=""):
        cmd = [sys.executable, os.path.abspath(__file__), "--out", a.out, "--worker", mode, "--reps", str(a.reps)] + (["--so", so] if so else [])
        r = subprocess.run(cmd, capture_output=True, text=True, cwd=ROOT)
        if r.returncode != 0:
            raise RuntimeError(f"{mode} {so}: {r.stderr[-3000:]}")
        return json.loads(r.stdout.strip().splitlines()[-1])

    res = {"card": card(), "workload": f"config 2: randomBouncing seed 42, {W}x675, {SPP} spp, depth {DEPTH}, AUTO, device-resident",
           "runs": a.runs, "timed_renders_per_run": a.reps}
    arms = {"default_branch": ("default", ""), "moments_off": ("moments_off", ""), "moments_on": ("moments_on", ""),
            "batched_500": ("batched", ""), "one_shot_500_moments": ("one_shot_moments", "")}
    if a.parent_so:
        arms["default_parent"] = ("default", a.parent_so)
    series = {k: [] for k in arms}
    for _ in range(a.runs):   # alternated: every arm once per round
        for k, (mode, so) in arms.items():
            series[k] += run(mode, so)
    res["to_noise"] = run("to_noise")
    res["card_after"] = card()
    for k, v in series.items():
        ms = sorted(x["ms"] for x in v)
        res[k] = {"ms": [x["ms"] for x in v], "ms_median": ms[len(ms) // 2], "ms_min": ms[0], "ms_max": ms[-1]}
        if "kernel_ms" in v[0]:
            res[k]["kernel_ms"] = [x["kernel_ms"] for x in v]
            res[k]["mpaths_s_median"] = W * 675 * SPP / (res[k]["ms_median"] * 1e-3) / 1e6
    os.makedirs(a.out, exist_ok=True)
    path = os.path.join(a.out, "progressive_probe.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
