#!/usr/bin/env python
"""bench.py — Mpaths/s of the rayz hot path on N B200s (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA backend
    python bench.py --impl reference --gpus N --steps K ...   # the reference algorithm on host cores
    python bench.py ... --dump-outputs DIR                    # also write the last timed step's frame to DIR/*.npy

A step is one full render of the workload (one pass of Tracer.render's pixel loop):
  N = 1 : BASELINE config 2 — RTOW final scene (randomBouncing, scene seed 42, 485 spheres),
          1200x675, 500 spp, max depth 50;
  N > 1 : BASELINE config 3 — same scene at 3840x2160, 1000 spp, image rows dealt to the ranks in
          round-robin bands of 4 rows, slabs gathered to GPU0 over NCCL (strong scaling).
`value`  : whole-job Mpaths/s with scene and camera resident in HBM, results left in HBM on GPU0.
`e2e`    : the same metric through the reference-facing C-ABI call with HOST buffers
           (rayz_cuda_upload_scene + rayz_cuda_render: H2D of the scene, D2H of linear float4 + RGB8).
`roofline`: the dominant kernel against BOTH roofs — algorithmic flop (SURVEY §8d / DESIGN.md) over its CUDA-event
           duration against the FFMA peak measured live by the K6 microbenchmark, and algorithmic HBM bytes over the same
           duration against MEASURED_PEAKS.json's copy bandwidth; `bound` names the nearer roof.
Only the cpu_baseline leg and --impl reference execute oracle/ (the CPU restatement of the Zig
reference, which cannot be compiled in this image).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "Mpaths/s"
ENTRY_BYTES = 64   # one queue entry of the staged K1 (rz_search.cuh: rz_queue_push)
NOMINAL_FP32_TFLOPS = 148 * 128 * 2 * 1.965e9 / 1e12  # 74.45: SMs x lanes x 2 flop x max SM clock
DUMP_BYTES = 60 << 20   # --dump-outputs: data bytes in all; with the .npy headers the files stay under 64 MB (10^6 bytes)


def dump_outputs(out_dir: str, frames: dict):
    """--dump-outputs: writes each [H, W, C] frame of the last timed step as out_dir/<name>.npy, float64 data as float64 and
    everything else as float32, so that two builds can be compared output for output.  When the frames would exceed
    DUMP_BYTES together, every file holds the same fixed, seeded sample of pixels instead: [n, C], pixels in row-major order."""
    os.makedirs(out_dir, exist_ok=True)
    import numpy as np
    frames = {k: np.asarray(v) for k, v in frames.items()}
    h, w = next(iter(frames.values())).shape[:2]
    as_dtype = {k: np.float64 if v.dtype == np.float64 else np.float32 for k, v in frames.items()}
    per_px = sum(np.dtype(as_dtype[k]).itemsize * v[0, 0].size for k, v in frames.items())
    pick = None
    if per_px * h * w > DUMP_BYTES:
        pick = np.sort(np.random.default_rng(0).choice(h * w, DUMP_BYTES // per_px, replace=False))
    for k, v in frames.items():
        assert v.shape[:2] == (h, w), (k, v.shape)
        out = v.astype(as_dtype[k])
        if pick is not None:
            out = out.reshape(h * w, -1)[pick]
        np.save(os.path.join(out_dir, k + ".npy"), out)
    print(f"bench.py: wrote {', '.join(k + '.npy' for k in frames)} to {out_dir}"
          + (f" ({len(pick)} of {h * w} pixels, seeded sample)" if pick is not None else ""), file=sys.stderr)


def workload(n_gpus: int, args) -> dict:
    if n_gpus <= 1:
        w = dict(name="config2: RTOW final scene (randomBouncing seed 42), 1200x675, 500 spp, depth 50",
                 width=1200, spp=500)
    else:
        w = dict(name="config3: RTOW final scene (randomBouncing seed 42), 3840x2160, 1000 spp, depth 50, "
                      "rows dealt to ranks in bands of 4", width=3840, spp=1000)
    if args.width:
        w["width"] = args.width
    if args.spp:
        w["spp"] = args.spp
    if args.width or args.spp:
        w["name"] = f"custom: randomBouncing seed 42, width {w['width']}, {w['spp']} spp, depth 50"
    w["height"] = int(float(w["width"]) / (16.0 / 9.0))
    w["depth"] = 50
    w["scene_seed"] = 42
    return w


# ------------------------------------------------------------------------------- clocks sampler
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows = []
        self.proc = None
        self.gpu = gpu_index
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        def pump():
            for line in self.proc.stdout:
                self.rows.append((time.time(), line.strip()))
        self.thread = threading.Thread(target=pump, daemon=True)
        self.thread.start()

    def stop(self, t0: float, t1: float) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        for ts, line in self.rows:
            if ts < t0 or ts > t1 + 0.2:
                continue
            f = [x.strip() for x in line.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------- reference arm
def run_reference(args, rank: int, world: int):
    """The reference algorithm (oracle port of the Zig renderer) on the box's host cores."""
    if rank != 0:
        return
    import oracle
    w = workload(args.gpus, args)
    threads = os.cpu_count() or 1
    scene = oracle.Scene.random_bouncing(w["scene_seed"])
    cam, h = oracle.default_camera(w["width"])
    assert h == w["height"]
    # bounded sample of the same workload: full resolution, few spp (the rate is spp-independent)
    # ~5 s of wall time per step at ~0.25 Mpaths/s per core
    spp = args.ref_spp or max(1, min(16, int(round(0.25e6 * threads * 5.0 / (w["width"] * h)))))
    paths = w["width"] * h * spp
    for i in range(args.warmup):
        scene.render(cam, w["width"], h, spp, w["depth"], seed=100 + i, threads=threads)
    t0 = time.perf_counter()
    for i in range(args.steps):
        img, _ = scene.render(cam, w["width"], h, spp, w["depth"], seed=200 + i, threads=threads)
    dt = (time.perf_counter() - t0) / args.steps
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"linear": img})
    v = paths / dt / 1e6
    sample = f"{w['width']}x{h} at {spp} spp of the {w['spp']}-spp workload per step (rate is spp-independent)"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": "Mpaths/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": w["name"], "width": w["width"], "height": h, "spp": w["spp"], "max_depth": w["depth"],
                   "paths_per_step": paths, "sample": sample, "sample_spp": spp,
                   "bounded_sample": "same scene, same resolution, same depth; each step renders sample_spp of the workload's spp "
                                     "(Mpaths/s does not depend on spp: every sample costs the same)"},
        "cpu_baseline": {"value": v, "unit": "Mpaths/s", "cores": threads, "kind": "port", "sample": sample,
                         "note": "oracle/ C++ restatement of the Zig reference (no zig toolchain in the image); rows "
                                 "over all host threads with per-row PRNG streams; the reference itself is single-threaded"},
        "e2e": {"value": v, "unit": "Mpaths/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }), file=_JSON_OUT, flush=True)


# ------------------------------------------------------------------------------- our arm
def algorithmic_flops_per_path(stats: dict, n_static: int, n_moving: int) -> dict:
    """SURVEY.md §8(d): F_path = sum over segments of the search flop + (S - p_sky)*F_shade + F_cam + p_sky*F_sky.

    A brute-force search costs F_isect = 16*n_static + 22*n_moving.  The staged K1 runs the camera
    segment of each path over a tile-culled list instead, so the search flop is scaled by the sphere tests the
    kernels actually counted (`sphere_tests`), not assumed to be segments * n_spheres.
    f_secondary = search flop of the segments after the first (what the dominant, persistent kernel does)."""
    paths = max(1, stats["paths"])
    S = stats["segments"] / paths
    p_sky = stats["ended_sky"] / paths
    n = max(1, n_static + n_moving)
    f_isect = n_static * 16 + n_moving * 22
    tests_per_path = stats["sphere_tests"] / paths if stats.get("sphere_tests") else S * n
    f_search = f_isect * tests_per_path / n + 18 * stats.get("node_tests", 0) / paths   # + box tests of the kernels that walk the BVH
    f_path = f_search + (S - p_sky) * 70 + 45 + p_sky * 19
    return {"segments_per_path": S, "p_sky": p_sky, "f_isect": f_isect, "f_path": f_path, "tests_per_path": tests_per_path,
            "f_secondary": max(0.0, S - 1.0) * f_isect}


def ncu_traffic_per_entry(kernel: str):
    """dram__bytes_read.sum + dram__bytes_write.sum of a kernel, per queue entry (= ray segment) it processed, from the committed
    `ncu --set full` capture of this round (profiles/traffic.json; the capture's launch is named there).  None if no capture."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            return json.load(f).get("dram_bytes_per_segment", {}).get(kernel)
    except Exception:
        return None


def measured_hbm_peak():
    """(GB/s, source) — MEASURED_PEAKS.json (driver-written) or the profiling recipe's fallback."""
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (torch copy, read+write bytes)"
    except Exception:
        return 6400.0, "fallback of B200_PROFILING.md (MEASURED_PEAKS.json absent)"


# The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints "NCCL version ..." to fd 1 when
# NCCL_DEBUG is set in the environment), so fd 1 is pointed at stderr for the life of the process and the JSON line
# goes to a private duplicate of the original stdout.
_JSON_OUT = None


def _claim_stdout():
    global _JSON_OUT
    if _JSON_OUT is None:
        sys.stdout.flush()
        _JSON_OUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)
    return _JSON_OUT


def main():
    _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--variant", default="auto", choices=["auto", "mega", "mega_single", "bvh", "wavefront"])
    ap.add_argument("--width", type=int, default=0, help="override workload width (quick checks only)")
    ap.add_argument("--spp", type=int, default=0, help="override workload spp (quick checks only)")
    ap.add_argument("--ref-spp", type=int, default=0, help="--impl reference: spp of the bounded sample")
    ap.add_argument("--rays-per-thread", type=int, default=0)
    ap.add_argument("--chunk", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-variants", action="store_true")
    ap.add_argument("--no-other-configs", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write the frame the last timed step computed to DIR/<name>.npy (float32 / float64, <= 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if args.gpus > 1 and world == 1 and "RANK" not in os.environ:
        # launched without torchrun: re-exec one rank per GPU the way the driver does
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}", "--master-addr",
               "127.0.0.1", "--master-port", "29541", os.path.abspath(__file__)] + sys.argv[1:]
        raise SystemExit(subprocess.call(cmd))
    if args.warmup < 3:
        args.warmup = 3  # timing rules: W >= 3

    import numpy as np
    import torch
    import torch.distributed as dist

    import rayz_b200
    from rayz_b200 import Backend

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the backend has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    ctl = None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        ctl = dist.new_group(backend="gloo")  # control-plane barriers that do not spin on the GPUs

    w = workload(world, args)
    W, H, SPP, DEPTH = w["width"], w["height"], w["spp"], w["depth"]
    tracer = rayz_b200.random_bouncing(W, seed=w["scene_seed"])   # host-side scene author (rayz.zig:45-168)
    scene = tracer.pool.arrays()
    cam = tracer.camera.rz

    be = Backend((local_rank,))
    if args.rays_per_thread or args.chunk:
        be.set_tuning(args.rays_per_thread, args.chunk)
    # a dedicated (non-default) torch stream: the library launches on it, torch events time it
    stream = torch.cuda.Stream(dev)
    torch.cuda.set_stream(stream)
    be.set_stream(stream.cuda_stream)
    be.upload_scene(scene)
    band = 4
    p = Backend.params(W, H, SPP, DEPTH, seed=1, variant=args.variant, shard_index=rank, shard_count=world, band_rows=band)
    rows_of = [int(be.lib.rayz_cuda_shard_rows(H, r, world, band)) for r in range(world)]
    my_rows = rows_of[rank]

    class DevArray:  # wraps a raw device pointer for torch.as_tensor (no copy)
        def __init__(self, ptr, shape, typestr):
            self.__cuda_array_interface__ = {"data": (ptr, False), "shape": shape, "typestr": typestr, "version": 3, "strides": None}

    from rayz_b200.dist import SlabGather
    gather_lin = SlabGather(H, (W, 4), torch.float32, dev, band) if world > 1 else None
    gather_rgb = SlabGather(H, (W, 3), torch.uint8, dev, band) if world > 1 else None

    last_frame = [None, None]   # device pointers of the latest step's linear and RGB8 frames (world == 1)

    def step_device():
        """One render, inputs resident in HBM, result left in HBM on GPU0 (after the NCCL gather for N>1)."""
        dl, d8, n = be.render_device(cam, p, sync=False)
        last_frame[:] = dl, d8
        if world == 1:
            return n
        lin = torch.as_tensor(DevArray(dl, (my_rows, W, 4), "<f4"), device=dev)
        rgb = torch.as_tensor(DevArray(d8, (my_rows, W, 3), "|u1"), device=dev)
        gather_lin.run(lin)      # slabs -> GPU0 over NCCL, interleaved into the full frame there
        gather_rgb.run(rgb)
        return n

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier(group=ctl)

    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    # ---- which kernel family the workload resolves to (RZ_VARIANT_AUTO picks by job size): one untimed render, then every
    # other pass names that variant explicitly, so the smaller stats pass counts the same kernels
    be.render_device(cam, p, sync=True)
    resolved = {1: "mega", 2: "wavefront", 3: "bvh", 4: "mega_single"}.get(be.timing()["variant"], args.variant)
    p = Backend.params(W, H, SPP, DEPTH, seed=1, variant=resolved, shard_index=rank, shard_count=world, band_rows=band)

    # ---- stats pass (not timed): segments/path for the algorithmic flop count
    ps = Backend.params(W, H, SPP, DEPTH, seed=1, variant=resolved, shard_index=rank, shard_count=world,
                        band_rows=band, collect_stats=True)
    be.render_device(cam, ps, sync=True)
    stats = be.stats()
    stage_stats = [be.stage_stats(k) for k in range(3)]
    tinfo = be.timing()

    # ---- warm-up
    for _ in range(args.warmup):
        step_device()
    barrier()

    # ---- timed: exactly K steps, CUDA events on the launching stream, L2 flushed between steps
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    barrier()
    t_wall0 = time.time()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    paths_step = 0
    for k in range(args.steps):
        flush_buf.zero_()
        ev[k][0].record(stream)
        paths_step = step_device()
        ev[k][1].record(stream)
        ev[k][1].synchronize()
    barrier()
    t_wall1 = time.time()
    step_ms = [a.elapsed_time(b) for a, b in ev]
    # the last timed step's frame, as a caller of the timed path receives it, before any later render reuses the buffers
    if args.dump_outputs and rank == 0:
        if world == 1:
            lin = torch.as_tensor(DevArray(last_frame[0], (H, W, 4), "<f4"), device=dev)
            rgb = torch.as_tensor(DevArray(last_frame[1], (H, W, 3), "|u1"), device=dev)
        else:
            lin, rgb = gather_lin.final, gather_rgb.final
        dump_outputs(args.dump_outputs, {"linear": lin.cpu().numpy(), "rgb8": rgb.cpu().numpy()})
    total_ms = torch.tensor([sum(step_ms)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
    total_ms = float(total_ms.item())
    clocks = sampler.stop(t_wall0, t_wall1) if rank == 0 else None
    total_paths = W * H * SPP
    ms_per_step = total_ms / args.steps
    value = total_paths / (ms_per_step * 1e-3) / 1e6

    # ---- path-kernel duration per launch (library CUDA events on the same stream), own pass
    # The staged K1 overlaps its passes on two streams; for clean per-kernel durations this pass asks for
    # serial passes (RZ_RENDER_SERIAL_PASSES): primary_ms = camera-segment kernels, kernel_ms - primary_ms = the
    # persistent secondary kernel (the dominant one).
    p_serial = Backend.params(W, H, SPP, DEPTH, seed=1, variant=resolved, shard_index=rank, shard_count=world, band_rows=band,
                              serial_passes=True)
    kms, pms, sms_, oms = [], [], [], []
    for _ in range(min(3, args.steps)):
        flush_buf.zero_()
        be.render_device(cam, p_serial, sync=True)
        kms.append(be.timing()["kernel_ms"])
        pms.append(be.timing()["primary_ms"])
        sms_.append(be.timing()["second_ms"])
        oms.append(be.timing()["sort_ms"])
    kt = torch.tensor([statistics.mean(kms), statistics.mean(pms), statistics.mean(sms_), statistics.mean(oms)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(kt, op=dist.ReduceOp.MAX)
    kern_ms, prim_ms, second_ms, sort_ms = (float(x) for x in kt.tolist())
    be.render_device(cam, p, sync=True)
    tinfo_run = be.timing()
    launches_per_step = be.timing()["launches"]
    passes_per_step = be.timing()["passes"]
    variant_ran = {1: "mega", 2: "wavefront", 3: "bvh", 4: "mega_single"}.get(be.timing()["variant"], "?")

    # ---- N > 1: (i) the gathered frame is checked, not just timed: at low spp the ranks' slabs, gathered over NCCL, must equal
    # the same frame rendered by rank 0 alone, byte for byte (counter-based RNG + integer accumulation: sharding-invariant);
    # (ii) rank 0 renders the FULL workload alone once, so that scaling can be read against the same work on one GPU.
    frame_check = single_gpu = None
    if world > 1:
        chk_spp = 4
        pc = Backend.params(W, H, chk_spp, DEPTH, seed=1, variant=resolved, shard_index=rank, shard_count=world, band_rows=band)
        dl, d8, _ = be.render_device(cam, pc, sync=True)
        lin = torch.as_tensor(DevArray(dl, (my_rows, W, 4), "<f4"), device=dev)
        rgb = torch.as_tensor(DevArray(d8, (my_rows, W, 3), "|u1"), device=dev)
        full_lin = gather_lin.run(lin)
        full_rgb = gather_rgb.run(rgb)
        barrier()
        if rank == 0:
            got_lin, got_rgb = full_lin.cpu().numpy().copy(), full_rgb.cpu().numpy().copy()
            p1 = Backend.params(W, H, chk_spp, DEPTH, seed=1, variant=resolved)
            ref_lin, ref_rgb, _ = be.render(cam, p1)
            import zlib
            frame_check = {"spp": chk_spp, "gathered_equals_single_gpu_render": bool(np.array_equal(got_lin, ref_lin) and np.array_equal(got_rgb, ref_rgb)),
                           "crc32_rgb8_gathered": zlib.crc32(got_rgb.tobytes()), "crc32_rgb8_single_gpu": zlib.crc32(ref_rgb.tobytes()),
                           "crc32_linear_gathered": zlib.crc32(got_lin.tobytes()), "crc32_linear_single_gpu": zlib.crc32(ref_lin.tobytes())}
            if not frame_check["gathered_equals_single_gpu_render"]:   # reported in the line, never hidden; the timing below still stands
                print("bench.py: WARNING: the gathered multi-GPU frame differs from the single-GPU render of the same seed", frame_check, file=sys.stderr)
            p_full = Backend.params(W, H, SPP, DEPTH, seed=1, variant=resolved)
            be.render_device(cam, p_full, sync=True)                     # warm-up (allocates this shape's buffers)
            ms1 = []
            for _ in range(2):
                flush_buf.zero_()
                a_ev, b_ev = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a_ev.record(stream)
                be.render_device(cam, p_full, sync=False)
                b_ev.record(stream)
                b_ev.synchronize()
                ms1.append(a_ev.elapsed_time(b_ev))
            single_gpu = {"value": total_paths / (min(ms1) * 1e-3) / 1e6, "unit": "Mpaths/s", "ms_per_step": min(ms1), "n_gpus": 1,
                          "workload": w["name"], "note": "rank 0 alone, whole frame, same kernels, device-resident (best of 2); "
                                                         "value / (n_gpus * this) is the strong-scaling efficiency on equal work"}
        barrier()

    # ---- the other BASELINE configs on one GPU (one warm-up + best of two timed renders each, device-resident; informational)
    other_configs = None
    if world == 1 and not args.no_other_configs:
        other_configs = {}
        for name, kw, ow, ospp in (("config4: 99,856 spheres (randomBouncing grid [-158,158)), device LBVH, 1920x1080, 256 spp, depth 50",
                                    dict(grid_lo=-158, grid_hi=158), 1920, 256),
                                   ("config5: glass-heavy (all-dielectric randomBouncing), 1200x675, 500 spp, depth 50", dict(glass_heavy=True), 1200, 500)):
            t_o = rayz_b200.random_bouncing(ow, seed=42, **kw)
            be_o = Backend((local_rank,))
            be_o.set_stream(stream.cuda_stream)
            be_o.upload_scene(t_o.pool.arrays())
            po = Backend.params(ow, t_o.img.h, ospp, DEPTH, seed=1, variant="auto")
            be_o.render_device(t_o.camera.rz, po, sync=True)
            best, info = None, None
            for _ in range(2):
                flush_buf.zero_()
                a_ev, b_ev = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a_ev.record(stream)
                be_o.render_device(t_o.camera.rz, po, sync=False)
                b_ev.record(stream)
                b_ev.synchronize()
                ms = a_ev.elapsed_time(b_ev)
                if best is None or ms < best:
                    best = ms
            be_o.render_device(t_o.camera.rz, po, sync=True)
            info = be_o.timing()
            npaths = ow * t_o.img.h * ospp
            other_configs[name.split(":")[0]] = {"workload": name, "value": npaths / (best * 1e-3) / 1e6, "unit": "Mpaths/s", "ms_per_step": best,
                                                 "paths_per_step": npaths, "spheres": len(t_o.pool.sphere_radius),
                                                 "variant": {1: "mega", 2: "wavefront", 3: "bvh", 4: "mega_single"}.get(info["variant"]),
                                                 "launches": info["launches"], "bvh_build_us": info["bvh_build_us"]}
            be_o.close()

    # ---- e2e: reference-facing call with host buffers (rank 0 drives all N GPUs through the
    # library's own multi-device context: this is what the single-process Zig host would call)
    e2e = None
    if not args.no_e2e:
        barrier()
        if rank == 0:
            be2 = Backend(tuple(range(world))) if world > 1 else be
            if args.rays_per_thread or args.chunk:
                be2.set_tuning(args.rays_per_thread, args.chunk)
            pe = Backend.params(W, H, SPP, DEPTH, seed=1, variant=args.variant)   # the call a user makes: AUTO unless overridden
            lin_h = torch.empty((H, W, 4), dtype=torch.float32).pin_memory().numpy()
            rgb_h = torch.empty((H, W, 3), dtype=torch.uint8).pin_memory().numpy()
            def step_e2e():
                be2.upload_scene(scene)
                return be2.render(cam, pe, out_linear=lin_h, out_rgb8=rgb_h)[2]
            for _ in range(2):
                step_e2e()
            t0 = time.perf_counter()
            for _ in range(args.steps):
                n = step_e2e()
            dt = (time.perf_counter() - t0) / args.steps
            e2e = {"value": n / dt / 1e6, "unit": "Mpaths/s", "ms_per_step": dt * 1e3,
                   "h2d_bytes_per_step": int(be2.scene_bytes + 152 + 56), "d2h_bytes_per_step": int(lin_h.nbytes + rgb_h.nbytes),
                   "api": "rayz_cuda_upload_scene + rayz_cuda_render (host buffers)" + (f", one process driving {world} GPUs, P2P gather" if world > 1 else "")}
            if world > 1:
                be2.close()
        barrier()

    # ---- the same workload with the opt-in pass size (RzTuning::queue_log2 = 28: twice the queue memory, half the passes; informational)
    tuned = None
    if world == 1 and not args.no_variants and resolved == "mega":
        be_t = Backend((local_rank,))
        be_t.set_stream(stream.cuda_stream)
        be_t.set_tuning(queue_log2=28)
        be_t.upload_scene(scene)
        be_t.render_device(cam, p, sync=True)
        ms_t = []
        for _ in range(3):
            flush_buf.zero_()
            a_ev, b_ev = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a_ev.record(stream)
            be_t.render_device(cam, p, sync=False)
            b_ev.record(stream)
            b_ev.synchronize()
            ms_t.append(a_ev.elapsed_time(b_ev))
        tuned = {"queue_log2": 28, "value": total_paths / (min(ms_t) * 1e-3) / 1e6, "unit": "Mpaths/s", "ms_per_step": min(ms_t),
                 "note": "not the default: 2^28-entry queues reserve ~72 GB for two passes instead of four (default 2^27: ~36 GB)"}
        be_t.close()

    # ---- the other kernel variants on the same workload (one timed render each; informational)
    variants = {}
    if world == 1 and not args.no_variants:
        for v in ("mega", "mega_single", "bvh", "wavefront"):
            pv = Backend.params(W, H, SPP, DEPTH, seed=1, variant=v)
            be.render_device(cam, pv, sync=True)
            flush_buf.zero_()
            be.render_device(cam, pv, sync=True)
            t = be.timing()
            variants[v] = {"mpaths_s": total_paths / (t["kernel_ms"] * 1e-3) / 1e6, "kernel_ms": t["kernel_ms"], "launches": t["launches"]}
            if v == "mega_single":   # the pure FP32-bound form: every segment searched by brute force in one kernel
                variants[v]["algorithmic_tflops"] = total_paths * (stats["segments"] / max(1, stats["paths"])) * (tinfo["n_static"] * 16 + tinfo["n_moving"] * 22) / (t["kernel_ms"] * 1e-3) / 1e12

    if rank == 0:
        fl = algorithmic_flops_per_path(stats, tinfo["n_static"], tinfo["n_moving"])
        # K6, the FP32 roof: three FFMA forms back to back, ~4 s each = 12 s of sustained FP32 load, SM clock sampled beside it
        k6_sampler = ClockSampler(local_rank)
        k6_sampler.start()
        time.sleep(0.2)
        k6_t0 = time.time()
        peak_tf, sms = be.fp32_peak(8000)
        k6_t1 = time.time()
        k6_clocks = k6_sampler.stop(k6_t0, k6_t1)
        hbm_peak, hbm_src = measured_hbm_peak()
        per_gpu_paths = total_paths / world
        two_stage = passes_per_step > 0
        stages = None
        if two_stage:
            # Staged K1: per-kernel durations from a render with serial passes (CUDA events around every launch, tails
            # included), algorithmic flop from each kernel's own sphere-test counter (16 per stationary, 22 per moving test;
            # shading flop left out: an undercount of < 1 %), algorithmic HBM bytes from the queue entries each kernel reads and
            # writes.  The roofline kernel is the one with the largest share of the step.
            scale = per_gpu_paths / max(1, stats["paths"])            # the stats pass covers this rank's share
            n_sph = max(1, tinfo["n_static"] + tinfo["n_moving"])
            f_test = fl["f_isect"] / n_sph                            # mean flop per sphere test of this scene
            meg_ms = kern_ms - prim_ms - second_ms - sort_ms
            n_stage = max(1, tinfo_run["sorted_stages"])
            ended = lambda st: st["ended_sky"] + st["ended_absorbed"] + st["ended_depth"]
            E, KEY, IDX = ENTRY_BYTES, 2, 4
            # queue entries written by a stage = its segments that did not end there; read by the next one
            out0 = (stage_stats[0]["segments"] - ended(stage_stats[0])) * scale          # primary -> first sorted stage
            in1 = stage_stats[1]["segments"] * scale                                      # all sorted stages, entries read
            out1 = (stage_stats[1]["segments"] - ended(stage_stats[1])) * scale           # ... entries written (next stage or tail)
            in2 = out1 - (in1 - out0) if n_stage else out0                                 # entries the tail kernel starts from
            in2 = max(0.0, in2)
            hbm = [out0 * (E + KEY) + 35 * W * H / world,                                 # primary: append entry + key (+ the frame, once)
                   in1 * (E + IDX) + out1 * E + (out1 - in2) * KEY,                       # sorted stages: gather entry through the index word (class bits inside), append entry (+ key)
                   in2 * E,                                                               # tail: read its entries
                   in1 * (2 * KEY + IDX)]                                                 # sort: keys read twice (count, scatter), index word written
            def stage(name, st, ms, launches, hbm_bytes):
                # a kernel that walked the BVH counted box tests too: 18 flop per box, 22 per (general) sphere test
                flop = 0.0
                if st is not None:
                    flop = (st["sphere_tests"] * 22 + st["node_tests"] * 18) * scale if st["node_tests"] else st["sphere_tests"] * scale * f_test
                d = {"kernel": name, "ms_per_step": ms, "launches_per_step": launches, "share_of_step": ms / kern_ms,
                     "flop": flop, "achieved_tflops": flop / (ms * 1e-3) / 1e12 if ms > 0 else None,
                     "frac": flop / (ms * 1e-3) / 1e12 / peak_tf if ms > 0 and peak_tf else None,
                     "hbm_bytes_algorithmic": hbm_bytes, "hbm_gbs": hbm_bytes / (ms * 1e-3) / 1e9 if ms > 0 else None,
                     "hbm_frac": hbm_bytes / (ms * 1e-3) / 1e9 / hbm_peak if ms > 0 else None}
                if st is not None:
                    d.update({"segments": st["segments"] * scale, "sphere_tests": st["sphere_tests"] * scale, "node_tests": st["node_tests"] * scale})
                return d
            stages = [stage("rz_primary_kernel (camera segments, tile-frustum cull)", stage_stats[0], prim_ms, passes_per_step, hbm[0]),
                      stage("rz_second_kernel (sorted segments 2.." + str(n_stage + 1) + ", per-unit cull)", stage_stats[1], second_ms, passes_per_step * n_stage, hbm[1]),
                      stage("rz_bvh_kernel<QUEUE> (persistent BVH kernel, later segments)" if stage_stats[2]["node_tests"] else
                            "rz_path_kernel<QUEUE> (persistent brute-force megakernel, later segments)", stage_stats[2], meg_ms, passes_per_step, hbm[2]),
                      stage("rz_bin_count_kernel + rz_bin_scan_kernel + rz_bin_scatter_kernel (key sort between the stages, rz_sort.cu)", None, sort_ms,
                            3 * passes_per_step * n_stage, hbm[3])]
            dom = max(stages[:3], key=lambda x: x["ms_per_step"])
            dom_name, dom_ms, dom_flop, dom_launches, dom_hbm = dom["kernel"], dom["ms_per_step"], dom["flop"], dom["launches_per_step"], dom["hbm_bytes_algorithmic"]
            dom_segments = dom["segments"]
            step_hbm = sum(hbm)
        else:
            dom_name = "rz_path_kernel (" + variant_ran + ")" if variant_ran != "bvh" else "rz_bvh_kernel"
            dom_ms = kern_ms
            dom_flop = per_gpu_paths * fl["f_path"]
            dom_launches = 1
            dom_hbm = step_hbm = 35 * W * H / world
            dom_segments = stats["segments"] * per_gpu_paths / max(1, stats["paths"])
        achieved = dom_flop / (dom_ms * 1e-3) / 1e12
        step_flops = per_gpu_paths * fl["f_path"] / (kern_ms * 1e-3) / 1e12
        fp32_frac = achieved / peak_tf if peak_tf else None
        hbm_gbs = dom_hbm / (dom_ms * 1e-3) / 1e9
        hbm_frac = hbm_gbs / hbm_peak
        tpe = ncu_traffic_per_entry(dom_name.split(" ")[0].split("<")[0])
        bound = "hbm" if hbm_frac > (fp32_frac or 0) else "fp32"
        # achieved / peak / unit / frac describe the roof named by `bound`; both roofs are spelled out beside them, per launch
        # (one launch = one kernel invocation; the dominant kernel is launched `launches_per_step` times per step)
        roofline = {"bound": bound, "kernel": dom_name,
                    "achieved": hbm_gbs if bound == "hbm" else achieved, "peak": hbm_peak if bound == "hbm" else peak_tf,
                    "unit": "GB/s" if bound == "hbm" else "TFLOP/s", "frac": hbm_frac if bound == "hbm" else fp32_frac,
                    "traffic": tpe * dom_segments / max(1, dom_launches) if tpe else None,
                    "traffic_note": "ncu dram__bytes_read.sum + dram__bytes_write.sum per launch, scaled per ray segment from the committed "
                                    "capture (profiles/traffic.json) — same unit and denominator as hbm.algorithmic_bytes_per_launch",
                    "fp32": {"achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s", "frac": fp32_frac,
                             "flop_per_launch": dom_flop / max(1, dom_launches),
                             "peak_source": "measured live: K6 FFMA/FFMA2 microbenchmark, 3 forms x ~4 s back to back, best form (MEASURED_PEAKS.json has no FP32 figure)",
                             "k6_clocks": k6_clocks, "frac_of_nominal": achieved / NOMINAL_FP32_TFLOPS, "nominal_peak": NOMINAL_FP32_TFLOPS},
                    "hbm": {"achieved": hbm_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": hbm_frac,
                            "algorithmic_bytes_per_launch": dom_hbm / max(1, dom_launches), "algorithmic_bytes_per_step": dom_hbm,
                            "entry_bytes": ENTRY_BYTES, "peak_source": hbm_src},
                    "kernel_ms_per_launch": dom_ms / max(1, dom_launches), "launches_per_step": dom_launches,
                    "kernel_ms_per_step": dom_ms, "share_of_step": dom_ms / kern_ms,
                    "stages": stages,
                    "all_kernels_ms_per_step_serial": kern_ms,
                    "whole_step": {"fp32_achieved": step_flops, "fp32_frac": step_flops / peak_tf if peak_tf else None,
                                   "hbm_bytes_algorithmic": step_hbm, "hbm_gbs": step_hbm / (kern_ms * 1e-3) / 1e9,
                                   "hbm_frac": step_hbm / (kern_ms * 1e-3) / 1e9 / hbm_peak},
                    "flop_per_path": fl["f_path"], "flop_per_path_dominant_kernel": dom_flop / per_gpu_paths,
                    "segments_per_path": fl["segments_per_path"], "sphere_tests_per_path": fl["tests_per_path"],
                    "flop_per_segment_search": fl["f_isect"],
                    "note": "The default (staged K1) wins by NOT doing arithmetic: tile-frustum and sorted-unit culls, and a BVH walk for the "
                            f"tail of the paths, cut the sphere tests per path from segments*n_spheres ({fl['segments_per_path'] * (tinfo['n_static'] + tinfo['n_moving']):.0f}) "
                            f"to {fl['tests_per_path']:.0f}, so its FP32 fraction is below that of K1 run as one brute-force "
                            "kernel, which variants.mega_single reports (frac_of_fp32_peak, the north star's 40 % target). "
                            "flop = algorithmic count of SURVEY 8(d) (16 per stationary, 22 per moving sphere test, 18 per BVH box test) of the "
                            "tests each kernel actually counted in a stats render of the same workload; tensor cores unused by design; "
                            "HBM bytes = the queue entries, keys and indices each kernel reads and writes (+ 35 B/pixel of framebuffer once per render)"}
        out = {
            "metric": METRIC, "value": value, "unit": "Mpaths/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": w["name"], "width": W, "height": H, "spp": SPP, "max_depth": DEPTH, "paths_per_step": total_paths,
                       "variant": variant_ran, "sharding": f"rows in bands of {band}, round-robin over {world} rank(s)",
                       "l2": "flushed between steps (256 MiB memset, untimed)"},
            "clocks": clocks, "gpu_launches": int(launches_per_step * args.steps),
            "roofline": roofline, "stats": {k: stats[k] for k in ("paths", "segments", "sphere_tests", "ended_sky", "ended_absorbed", "ended_depth")},
        }
        if e2e:
            out["e2e"] = e2e
        if frame_check:
            out["frame_check"] = frame_check
        if single_gpu:
            out["single_gpu_same_workload"] = single_gpu
            out["strong_scaling_efficiency_same_workload"] = value / (world * single_gpu["value"])
        if other_configs:
            out["other_configs"] = other_configs
        if tuned:
            out["tuned"] = tuned
        if variants:
            if "mega_single" in variants and peak_tf:
                variants["mega_single"]["frac_of_fp32_peak"] = variants["mega_single"]["algorithmic_tflops"] / peak_tf
            out["variants"] = variants
        if not args.no_cpu_baseline and world == 1:
            import oracle
            sc = oracle.Scene.random_bouncing(w["scene_seed"])
            ocam, oh = oracle.default_camera(W)
            spp_cpu = 3
            t0 = time.perf_counter()
            sc.render(ocam, W, oh, spp_cpu, DEPTH, seed=5, threads=1)
            dt = time.perf_counter() - t0
            out["cpu_baseline"] = {"value": W * oh * spp_cpu / dt / 1e6, "unit": "Mpaths/s", "cores": 1, "kind": "port",
                                   "sample": f"{W}x{oh} at {spp_cpu} spp, 1 thread, one sequential PRNG (the reference's own structure)",
                                   "seconds": dt}
        print(json.dumps(out), file=_JSON_OUT, flush=True)
    if world > 1:
        dist.barrier(group=ctl)
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
