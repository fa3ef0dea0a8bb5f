"""Cost of the ID mattes (rayz_cuda_render_mattes) next to the guide buffers, one JSON file.

    python scripts/mattes_probe.py --out OUT_DIR [--runs 7] [--profile]

With the card's name, power limit and max SM clock read in the same call, it times config 2 (1200x675, randomBouncing seed 42,
render seed 1) at 16, 64, 256 and 1024 spp: Backend.mattes with 6 ranks and Backend.guides over the same samples, alternated,
host wall time of each call (it ends in a device synchronise; the copies out are included), medians after one warm-up call
of each.  Then config 4 (99,856 spheres, device LBVH) at 64 spp.  --profile adds a torch.profiler capture of one mattes call
and one guides call at 64 spp on config 2 (a run of its own: tracing slows the host), kernel times by name.
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
    ap.add_argument("--profile", action="store_true")
    a = ap.parse_args()
    sys.path.insert(0, ROOT)
    import numpy as np

    import rayz_b200
    from rayz_b200 import Backend

    def timed(fn):
        t0 = time.perf_counter()
        fn()
        return (time.perf_counter() - t0) * 1e3

    res = {"card": card(), "configs": []}
    for name, kw, w, spps in (("config2", {}, 1200, (16, 64, 256, 1024)),
                              ("config4", {"grid_lo": -158, "grid_hi": 158}, 1200, (64,))):
        t = rayz_b200.random_bouncing(w, seed=42, **kw)
        be = Backend((0,))
        be.upload_scene(t.pool.arrays())
        cam, h = t.camera.rz, t.img.h
        for spp in spps:
            p = Backend.params(w, h, spp, 50, seed=1)
            be.mattes(cam, p, 6)
            be.guides(cam, p)
            m, g = [], []
            for _ in range(a.runs):
                m.append(timed(lambda: be.mattes(cam, p, 6)))
                g.append(timed(lambda: be.guides(cam, p)))
            row = {"scene": name, "width": w, "height": h, "spp": spp, "mattes_ms": float(np.median(m)), "guides_ms": float(np.median(g)),
                   "mattes_all_ms": m, "guides_all_ms": g}
            row["ratio"] = row["mattes_ms"] / row["guides_ms"]
            print(json.dumps({k: v for k, v in row.items() if not k.endswith("all_ms")}), flush=True)
            res["configs"].append(row)
        if a.profile and name == "config2":
            import torch
            from torch.profiler import ProfilerActivity, profile
            p = Backend.params(w, h, 64, 50, seed=1)
            with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
                be.mattes(cam, p, 6)
                be.guides(cam, p)
                torch.cuda.synchronize()
            ks = {}
            for e in prof.events():
                if e.device_type == torch.autograd.DeviceType.CUDA:
                    ks[e.name] = ks.get(e.name, 0.0) + e.device_time / 1e3
            res["profile_64spp_ms"] = ks
            print(json.dumps(ks), flush=True)
        be.close()
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "mattes_probe.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(res["card"])


if __name__ == "__main__":
    main()
