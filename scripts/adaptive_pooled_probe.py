"""What pooled adaptive stopping (RZ_RENDER_ADAPTIVE_POOLED) buys and costs, against plain adaptive and uniform doubling, one
JSON file.

    python scripts/adaptive_pooled_probe.py --out OUT_DIR [--quick]

With the card's name and power limit read in the same call (depth 50, BVH variant, start 4 and 16 spp, cap 4096):
  * honesty and cost at 1200 x 675 on config 2 and penultimate_scene, targets 2/255 and 1/255, under Philox, Sobol and RQMC:
    the measured rms displayed error over the non-capped pixels (overall and per group of pixels with the same final count),
    paths and wall time of pooled adaptive, plain adaptive and uniform doubling to the same max estimate (render +
    rayz_cuda_noise per batch).  The measured error is rqmc_probe.py's: against a 16384-spp Philox reference made of two
    8192-spp halves, the reference's own noise removed.  Wall time: host clock around calls that end in a device synchronise,
    the three arms alternated after one warm-up call of each;
  * the NU0 sweep (0 = the plain rule, 4, 8, 16, 32, 64) on held-out scenes: config 5 (glass-heavy) and config 2 with render
    seed 61, both 1200 x 675.  NU0 is a compile-time constant, so the sweep replays the stopping rule in numpy f64 on a ladder of
    uniform frames (counts 4, 8, ..., 4096 of the same samples): a pixel with c samples equals the same pixel of a uniform c-spp
    render bit for bit, so the replay needs only each frame's linear and out_err (u = n e^2).  The replay at the compiled NU0 is
    checked against the library's own counts (the agreement is recorded);
  * the segment pass's device time (torch.profiler, a pass of its own) with the gain alone, the prior alone and both.
"""
from __future__ import annotations

import argparse
import json
import os
import re
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SAMPLERS = {"philox": {}, "sobol": {"sobol": True}, "rqmc": {"sobol": True, "rqmc": True}}
SWEEP = (0, 4, 8, 16, 32, 64)


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else f"nvidia-smi failed: {r.stderr.strip()}"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--quick", action="store_true", help="320 x 180 and fewer arms: a rehearsal of the script")
    a = ap.parse_args()
    sys.path.insert(0, ROOT)
    import numpy as np
    import rayz_b200
    from rayz_b200 import Backend

    nu0_lib = float(re.search(r"NU0 = (\d+)", open(os.path.join(ROOT, "include", "rayz_cuda.h")).read()).group(1))
    W = 320 if a.quick else 1200
    REF = 1024 if a.quick else 8192
    CAP = 4096
    res = {"card": card(), "width": W, "nu0_compiled": nu0_lib}
    luma = lambda x: 0.2126 * x[..., 0] + 0.7152 * x[..., 1] + 0.0722 * x[..., 2]
    disp = lambda x: np.sqrt(np.maximum(luma(x), 1e-4))

    def setup(name):
        t = {"config2": lambda: rayz_b200.random_bouncing(W, seed=42), "config5": lambda: rayz_b200.random_bouncing(W, seed=42, glass_heavy=True),
             "penultimate": lambda: rayz_b200.penultimate_scene(W)}[name]()
        h = int(W / rayz_b200.ASPECT_RATIO)
        b = Backend((0,))
        b.upload_scene(t.pool.arrays())
        cam = t.camera.rz
        ra, _, _ = b.render(cam, Backend.params(W, h, REF, 50, seed=1001, variant="bvh"), want_rgb8=False)
        rc, _, _ = b.render(cam, Backend.params(W, h, REF, 50, seed=1002, variant="bvh"), want_rgb8=False)
        ra, rc = ra[..., :3].astype(np.float64), rc[..., :3].astype(np.float64)
        return dict(b=b, cam=cam, h=h, ref=disp((ra + rc) / 2), ref_noise=(disp(ra) - disp(rc)) ** 2 / 4)

    def measured(S, lin, mask):
        d2 = (disp(lin[..., :3].astype(np.float64)) - S["ref"]) ** 2 - S["ref_noise"]
        return float(np.sqrt(max(d2[mask].mean(), 0.0))) if mask.any() else None

    def honesty(S, lin, counts, target):
        live = counts < CAP
        groups = {}
        for c in np.unique(counts[live]):
            m = counts == c
            if m.sum() >= 2000:
                groups[int(c)] = {"pixels": int(m.sum()), "ratio": measured(S, lin, m) / target}
        r = measured(S, lin, live)
        return {"ratio": None if r is None else r / target, "capped": int((~live).sum()), "groups": groups}

    # ---- honesty and cost of the library's three arms
    arms = {}
    scenes = ("config2", "penultimate")
    targets = (2, 1)
    starts = (4, 16)
    samplers = ("philox", "rqmc") if a.quick else tuple(SAMPLERS)
    for name in scenes:
        S = setup(name)
        b, cam, h = S["b"], S["cam"], S["h"]
        for ts in targets:
            target = ts / 255
            for start in starts:
                for s in samplers:
                    p = Backend.params(W, h, start, 50, seed=61, variant="bvh", **SAMPLERS[s])

                    def pooled():
                        lin, _, paths, nz = b.render_to_noise(cam, p, target, CAP, adaptive=True, pooled=True)
                        return lin, paths, nz, b.pixel_samples()

                    def plain():
                        lin, _, paths, nz = b.render_to_noise(cam, p, target, CAP, adaptive=True)
                        return lin, paths, nz, b.pixel_samples()

                    def uniform():
                        q = Backend.params(W, h, start, 50, seed=61, variant="bvh", moments=True, **SAMPLERS[s])
                        lin, _, _ = b.render(cam, q, want_rgb8=False)
                        n, nz = start, b.noise(target)[1]
                        while nz["max_err"] > target and n < CAP:
                            q = Backend.params(W, h, min(n, CAP - n), 50, seed=61, sample_offset=n, variant="bvh", accumulate=True, moments=True,
                                               **SAMPLERS[s])
                            lin, _, _ = b.render(cam, q, want_rgb8=False)
                            n += q.spp
                            nz = b.noise(target)[1]
                        return lin, n * W * h, nz, np.full((h, W), n, dtype=np.uint32)

                    fns = {"pooled": pooled, "plain": plain, "uniform_to_max": uniform}
                    for f in fns.values():
                        f()                                          # warm-up of the same shapes
                    times = {k: [] for k in fns}
                    out = {}
                    for _ in range(1 if a.quick else 2):
                        for k, f in fns.items():
                            t0 = time.perf_counter()
                            out[k] = f()
                            times[k].append(time.perf_counter() - t0)
                    for k, (lin, paths, nz, counts) in out.items():
                        row = {"paths": int(paths), "wall_ms": [1e3 * x for x in times[k]], "samples": nz["samples"], "max_estimate": nz["max_err"],
                               "n_above": nz["n_above"], "mean_spp": float(counts.mean())}
                        row.update(honesty(S, lin, counts, target))
                        key = f"{name}_{ts}/255_start{start}_{s}_{k}"
                        arms[key] = row
                        print(key, {x: y for x, y in row.items() if x != "groups"}, flush=True)
        b.close()
    res["arms"] = arms

    # ---- the NU0 sweep by replay, on held-out scenes (Philox and Sobol: the iid estimate, which a uniform frame shows exactly)
    def ladder(S, s):
        b, cam, h = S["b"], S["cam"], S["h"]
        frames = {}
        q = Backend.params(W, h, 4, 50, seed=61, variant="bvh", moments=True, **SAMPLERS[s])
        lin, _, _ = b.render(cam, q, want_rgb8=False)
        n = 4
        while True:
            frames[n] = (lin[..., :3].copy(), b.noise()[0].astype(np.float64))
            if n >= CAP:
                break
            q = Backend.params(W, h, n, 50, seed=61, sample_offset=n, variant="bvh", accumulate=True, moments=True, **SAMPLERS[s])
            lin, _, _ = b.render(cam, q, want_rgb8=False)
            n *= 2
        return frames

    def replay(frames, start, target, nu0, h):
        nseg = -(-W // 64)
        seg = (np.arange(h)[:, None] * nseg + np.arange(W)[None, :] // 64).ravel()
        uof = {c: (c * e * e).ravel() for c, (_, e) in frames.items()}
        counts = np.full(h * W, start)
        frozen = np.zeros(h * W)
        tgt = float(np.float32(target))

        def segment_pass(n):
            d = counts - 1.0
            u = np.empty(h * W)
            for c in np.unique(counts):
                m = counts == c
                u[m] = uof[int(c)][m]
            num = np.bincount(seg, d * u, h * nseg)
            den = np.bincount(seg, d, h * nseg)
            U = np.where(den > 0, num / np.where(den > 0, den, 1), 0.0)
            top = counts == n
            frozen[top] = U[seg[top]]
            return u

        n = start
        while n < CAP:
            u = segment_pass(n)
            e = np.sqrt((nu0 * frozen + (counts - 1) * u) / (nu0 + counts - 1) / counts).astype(np.float32).astype(np.float64)
            act = (counts == n) & (e > tgt)
            if not act.any():
                break
            b_ = min(n, CAP - n)
            counts[act] += b_
            n += b_
        u = segment_pass(n)
        lin = np.empty((h * W, 3))
        for c in np.unique(counts):
            m = counts == c
            lin[m] = frames[int(c)][0].reshape(-1, 3)[m]
        return counts.reshape(h, W), lin.reshape(h, W, 3)

    sweep = {}
    for name in ("config5", "config2_seed61"):
        S = setup(name.split("_")[0])
        h = S["h"]
        for s in (("philox",) if a.quick else ("philox", "sobol")):
            frames = ladder(S, s)
            for ts in targets:
                target = ts / 255
                for start in starts:
                    for nu0 in SWEEP:
                        counts, lin = replay(frames, start, target, nu0, h)
                        row = {"paths": int(counts.sum()), "mean_spp": float(counts.mean())}
                        row.update(honesty(S, lin, counts, target))
                        key = f"{name}_{s}_{ts}/255_start{start}_nu0={nu0}"
                        sweep[key] = row
                        print(key, {x: y for x, y in row.items() if x != "groups"}, flush=True)
                    # the replay against the library at the compiled NU0
                    p = Backend.params(W, h, start, 50, seed=61, variant="bvh", **SAMPLERS[s])
                    S["b"].render_to_noise(S["cam"], p, target, CAP, adaptive=True, pooled=True)
                    lib_counts = S["b"].pixel_samples()
                    counts, _ = replay(frames, start, target, nu0_lib, h)
                    sweep[f"{name}_{s}_{ts}/255_start{start}_replay_agreement"] = float((lib_counts == counts).mean())
                    print("replay agreement", name, s, ts, start, sweep[f"{name}_{s}_{ts}/255_start{start}_replay_agreement"], flush=True)
        S["b"].close()
    res["nu0_sweep"] = sweep

    # ---- the segment pass's device time
    import torch
    from torch.profiler import ProfilerActivity, profile
    t = rayz_b200.random_bouncing(W, seed=42)
    b = Backend((0,))
    b.upload_scene(t.pool.arrays())
    cam, h = t.camera.rz, int(W / rayz_b200.ASPECT_RATIO)
    seg = {}
    for label, kw, pooled in (("gain", SAMPLERS["rqmc"], False), ("prior", {}, True), ("gain+prior", SAMPLERS["rqmc"], True)):
        p = Backend.params(W, h, 4, 50, seed=1, variant="bvh", **kw)
        b.render_to_noise(cam, p, 1 / 255, 4, adaptive=True, pooled=pooled)   # one round: the frame the pass reads
        b.noise()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(20):
                b.noise()
        ev = [e for e in prof.events() if "rz_segment_kernel" in e.name]
        seg[label] = {"calls": len(ev), "mean_us": float(np.mean([e.device_time for e in ev])) if ev else None}
        print("segment pass", label, seg[label], flush=True)
    res["segment_pass"] = seg
    b.close()

    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "adaptive_pooled_probe.json"), "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", os.path.join(a.out, "adaptive_pooled_probe.json"))


if __name__ == "__main__":
    main()
