"""What rendering many small views in one frame buys (yr_set_cameras): three arms over the same pixel count, per workload.

  (a) batch    one renderer, V orbit cameras of W x H set with yr_set_cameras, one render of all views;
  (b) loop     the same V cameras rendered one after the other by one renderer (scene uploaded once);
  (c) single   one camera at sqrt(V) W x sqrt(V) H: the same pixel count in one frame.

Workloads: bench.py's C2 soup (depth 1) and its McLaren-shaped scene (full paths), default traversal.  Every render is one
wave of `spp` samples; the arms alternate (rotating order), after warm-up renders of each.  Times are host clocks around
yr_render_sync (the frame's device work is done when it returns; frames stay on the device), medians over the timed
rounds; Mrays/s counts the reference's rays (YcStats.raysReference).  Each view of (a) and (b) is hashed and must match.
--profile adds a torch.profiler run (separate from the timing) of one render of (a) and the V renders of (b): kernel time
per kernel name, and the share of the wall time the GPU ran a kernel.  Prints one JSON object with the GPU's name and
power limit read in the same run; --out also writes it.

  python tools/multiview_bench.py [--views 64] [--size 256] [--spp 4] [--rounds 5] [--profile] [--out profiles/r03_multiview.json]"""
import argparse
import hashlib
import json
import math
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

import bench  # noqa: E402  (the workloads exactly as the benchmark builds them)
import yart_b200 as Y  # noqa: E402
from yart_b200 import capi  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    name, limit = (q.stdout.strip().split(", ") + ["?", "?"])[:2]
    return dict(gpu=name, power_limit=limit)


def orbit(views, w, h):
    """`views` cameras on a horizontal circle around the workload camera's target, at its distance and height."""
    pos, target = np.asarray(bench.CAM["pos"], np.float64), np.asarray(bench.CAM["target"], np.float64)
    d = pos - target
    radius, height = math.hypot(d[0], d[2]), d[1]
    phase = math.atan2(d[0], d[2])
    cams = []
    for k in range(views):
        a = phase + 2.0 * math.pi * k / views
        p = target + np.array([radius * math.sin(a), height, radius * math.cos(a)])
        cams.append(Y.make_camera(w, h, bench.CAM["focal"], bench.CAM["fnum"], tuple(p), tuple(target), (0, 0, 0), bench.CAM["exposure"]))
    return cams


def digest(a):
    return hashlib.sha1(np.ascontiguousarray(a).tobytes()).hexdigest()[:12]


def renderer(scene, w, h, cam, spp):
    return Y.Renderer(w, h, cam, scene, samples=spp, first_wave_samples=spp, max_wave_samples=spp, max_depth=bench.MAX_DEPTH,
                      traversal=Y.TRAVERSAL_AUTO)


def measure(workload, views, size, spp, rounds, warmup, profile):
    n_tris = bench.DEFAULT_TRIS[workload]
    bench.select_workload(workload, n_tris)
    scene = Y.Scene(bench.scene_path(n_tris, workload))
    cams = orbit(views, size, size)
    side = int(round(math.sqrt(views))) * size
    batch = renderer(scene, size, size, cams, spp)
    loop = renderer(scene, size, size, cams[0], spp)
    single = renderer(scene, side, side, orbit(1, side, side)[0], spp)

    def run_batch():
        return batch.render_sync()["total_rays"]

    def run_loop():
        rays = 0
        for cam in cams:
            loop.set_camera(cam)
            rays += loop.render_sync()["total_rays"]
        return rays

    def run_single():
        return single.render_sync()["total_rays"]

    arms = dict(batch=run_batch, loop=run_loop, single=run_single)
    ms = {k: [] for k in arms}
    rays = {}
    names = list(arms)
    for r in range(warmup + rounds):
        for k in names[r % 3:] + names[:r % 3]:
            t0 = time.perf_counter()
            rays[k] = arms[k]()
            dt = (time.perf_counter() - t0) * 1e3
            if r >= warmup:
                ms[k].append(dt)
    out = dict(workload=bench.WORKLOAD_TEXT.replace(f"{bench.W}x{bench.H}", "see arms"), spp=spp, rounds=rounds)
    for k in names:
        med = statistics.median(ms[k])
        out[k] = dict(ms=round(med, 3), ms_min=round(min(ms[k]), 3), mrays_per_s=round(rays[k] / med / 1e3, 1), rays=int(rays[k]))
    out["batch"]["what"] = f"{views} views of {size}x{size} in one frame (yr_set_cameras)"
    out["loop"]["what"] = f"the same {views} cameras one after the other, one renderer"
    out["single"]["what"] = f"one camera at {side}x{side}"
    out["batch_over_single"] = round(out["batch"]["mrays_per_s"] / out["single"]["mrays_per_s"], 3)
    out["batch_over_loop"] = round(out["batch"]["mrays_per_s"] / out["loop"]["mrays_per_s"], 3)

    # every view of the batch against the same camera rendered alone
    run_batch()
    hdr_batch = batch.read(want_ldr=False)[0]
    hashes_batch = [digest(hdr_batch[v]) for v in range(views)]
    hashes_loop = []
    for cam in cams:
        loop.set_camera(cam)
        loop.render_sync()
        hashes_loop.append(digest(loop.read(want_ldr=False)[0]))
    out["view_hashes_batch"], out["view_hashes_loop"] = hashes_batch, hashes_loop
    out["views_match"] = hashes_batch == hashes_loop

    if profile:
        out["profile"] = dict(batch=profiled(run_batch), loop=profiled(run_loop))
    for r in (batch, loop, single):
        r.close()
    return out


def profiled(fn):
    """Kernel time per kernel name over one call of `fn`, its launch count, and the GPU-busy share of the wall time."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        t0 = time.perf_counter()
        fn()
        wall_ms = (time.perf_counter() - t0) * 1e3
    kernels = {}
    busy = []
    for e in prof.events():
        if e.device_type != torch.autograd.DeviceType.CUDA or "memcpy" in e.name.lower() or "memset" in e.name.lower():
            continue
        k = kernels.setdefault(e.name[:80], dict(launches=0, ms=0.0))
        k["launches"] += 1
        k["ms"] += e.device_time / 1e3
        busy.append((e.time_range.start, e.time_range.end))
    busy.sort()
    covered, end = 0.0, -1.0
    for s, e in busy:  # union of the kernels' intervals (the two lanes' kernels overlap)
        if e > end:
            covered += e - max(s, end)
            end = e
    top = sorted(kernels.items(), key=lambda kv: -kv[1]["ms"])[:12]
    return dict(wall_ms=round(wall_ms, 3), kernel_launches=sum(k["launches"] for k in kernels.values()),
                gpu_busy_ms=round(covered / 1e3, 3), gpu_busy_share=round(covered / 1e3 / wall_ms, 3),
                kernels={n: dict(launches=k["launches"], ms=round(k["ms"], 3)) for n, k in top})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--views", type=int, default=64)
    ap.add_argument("--size", type=int, default=256)
    ap.add_argument("--spp", type=int, default=4)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--workloads", default="soup,mclaren")
    ap.add_argument("--profile", action="store_true")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    Y.use_library(capi.load())
    rec = dict(gpu_info(), timing="host clock around yr_render_sync (one wave per render), median over rounds, arms alternating")
    for wl in args.workloads.split(","):
        rec[wl] = measure(wl, args.views, args.size, args.spp, args.rounds, args.warmup, args.profile)
    text = json.dumps(rec, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
