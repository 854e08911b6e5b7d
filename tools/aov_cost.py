"""What the first-hit AOVs (yc_enable_aovs) cost per wave: bench.py's C2 (1 M-triangle soup, 1920x1080, waves of 4 samples,
depth 1) and its Sponza-shaped full-path workload, each rendered by two contexts of the same scene — AOVs off and on —
whose waited-for waves (yc_render_wave) alternate, ABBA, so that drift of the shared box falls on both arms alike.
Prints one JSON object (ms per wave, overhead, GPU name and power limit read in the same run); --out also writes it.

  python tools/aov_cost.py [--waves 24] [--out profiles/r03_aov_cost.json]"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402  (the workloads exactly as the benchmark builds them)
import yart_b200 as Y  # noqa: E402
from yart_b200 import capi  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    name, limit = (q.stdout.strip().split(", ") + ["?", "?"])[:2]
    return dict(gpu=name, power_limit=limit)


def measure(workload, waves, spp):
    n_tris = bench.DEFAULT_TRIS[workload]
    bench.select_workload(workload, n_tris)
    scene = Y.Scene(bench.scene_path(n_tris, workload))
    cam = Y.make_camera(bench.W, bench.H, bench.CAM["focal"], bench.CAM["fnum"], bench.CAM["pos"], bench.CAM["target"], (0, 0, 0),
                        bench.CAM["exposure"])
    arms = {}
    for on in (False, True):
        ctx = Y.Context(max_depth=bench.MAX_DEPTH, traversal=Y.TRAVERSAL_AUTO)
        ctx.upload_scene(scene)
        ctx.set_camera(cam)
        if on:
            ctx.enable_aovs()
        ctx.begin_frame(bench.W, bench.H, spp * (waves + 3), 64, (0, 0, 0), Y.TONEMAP_AGX)
        arms[on] = ctx
    times = {False: [], True: []}
    for k in range(waves + 3):  # 3 warm-up waves per arm
        for on in ((False, True) if k % 2 == 0 else (True, False)):
            t0 = time.perf_counter()
            arms[on].render_wave(k * spp, spp, k * spp)
            dt = (time.perf_counter() - t0) * 1e3
            if k >= 3:
                times[on].append(dt)
    off_ms, on_ms = statistics.median(times[False]), statistics.median(times[True])
    for ctx in arms.values():
        ctx.close()
    return dict(workload=bench.WORKLOAD_TEXT, waves_per_arm=waves, spp_per_wave=spp, ms_per_wave_off=round(off_ms, 3),
                ms_per_wave_on=round(on_ms, 3), overhead_pct=round(100.0 * (on_ms / off_ms - 1.0), 2),
                ms_off_min=round(min(times[False]), 3), ms_on_min=round(min(times[True]), 3))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--waves", type=int, default=24, help="timed waves per arm (at least 20)")
    ap.add_argument("--spp", type=int, default=4)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    Y.use_library(capi.load())
    rec = dict(gpu_info(), timing="host clock around yc_render_wave (returns after the wave's device work), median over waves",
               c2=measure("soup", args.waves, args.spp), sponza=measure("sponza", args.waves, args.spp))
    text = json.dumps(rec, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
