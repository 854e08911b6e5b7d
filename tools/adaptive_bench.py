"""What adaptive sampling (yr_set_adaptive) buys: time, mean samples per pixel and HDR error against a converged render.

Workloads: bench.py's Sponza-shaped and McLaren-shaped scenes at 1920x1080, full paths, default traversal, the renderer's
default wave schedule (64, then 128 per wave).  Arms per workload:
  off      non-adaptive renders of 256, 512, 768 and 1024 samples;
  t=...    1024-sample renders with adaptive sampling at each threshold (minSamples 64, lumaFloor 1e-3);
against a non-adaptive render of 4096 samples.  Time: host clock around yr_render_sync (it returns after the device work);
every arm runs --repeats times, the arms in a rotated order each round, and the median, minimum and maximum are reported.
mean_spp: ΣS / pixels (yr_read_adaptive).  rel_mse: bench.rel_mse of the HDR frame against the reference's (the frames
are deterministic: the same in every round).
Then the per-wave cost of the machinery with threshold 0 (nothing stops, the same frame) against off, on bench.py's C2
step (the 1 M-triangle soup at 1080p, depth 1, 4-sample waves through yc_render_wave), A and B alternating on one card;
the two frames must be identical.  Prints one JSON object with the GPU's name and power limit read in the same run;
--out also writes it.

  python tools/adaptive_bench.py [--spp 1024] [--ref-spp 4096] [--repeats 3] [--c2-waves 40] [--c2-rounds 7]
                                 [--out profiles/r03_adaptive.json]"""
import argparse
import json
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

THRESHOLDS = [0.1, 0.05, 0.02, 0.01]
MIN_SAMPLES, LUMA_FLOOR = 64, 1e-3


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    name, limit = (q.stdout.strip().split(", ") + ["?", "?"])[:2]
    return dict(gpu=name, power_limit=limit)


def render(scene, spp, adaptive=None):
    cam = Y.make_camera(bench.W, bench.H, bench.CAM["focal"], bench.CAM["fnum"], bench.CAM["pos"], bench.CAM["target"], (0, 0, 0),
                        bench.CAM["exposure"])
    r = Y.Renderer(bench.W, bench.H, cam, scene, samples=spp, max_depth=bench.MAX_DEPTH, traversal=Y.TRAVERSAL_AUTO, adaptive=adaptive)
    t0 = time.perf_counter()
    d = r.render_sync()
    ms = (time.perf_counter() - t0) * 1e3
    hdr, _, st = r.read(want_ldr=False)
    mean_spp = float(r.read_adaptive()["samples"].astype(np.float64).mean()) if adaptive else float(spp)
    r.close()
    return hdr, dict(ms=round(ms, 1), mean_spp=round(mean_spp, 2), samples_taken=d["samples_taken"], rays=d["total_rays"])


def quality(workload, spp, ref_spp, repeats):
    n_tris = bench.DEFAULT_TRIS[workload]
    bench.select_workload(workload, n_tris)
    scene = Y.Scene(bench.scene_path(n_tris, workload))
    render(scene, 64)  # warm-up: modules, allocations
    ref, ref_rec = render(scene, ref_spp)
    arms = [(f"off {s}", s, None) for s in (spp // 4, spp // 2, 3 * spp // 4, spp)]
    arms += [(f"t={t}", spp, (t, MIN_SAMPLES, LUMA_FLOOR)) for t in THRESHOLDS]
    rows = {}
    for r in range(repeats):
        k = r % len(arms)
        for name, s, adaptive in arms[k:] + arms[:k]:
            hdr, rec = render(scene, s, adaptive)
            err = bench.rel_mse(hdr, ref)
            if name not in rows:
                rows[name] = dict(arm=name, rel_mse=err, mean_spp=rec["mean_spp"], samples_taken=rec["samples_taken"], rays=rec["rays"],
                                  ms_runs=[])
            assert rows[name]["rel_mse"] == err and rows[name]["rays"] == rec["rays"], f"{workload} {name}: frames differ between rounds"
            rows[name]["ms_runs"].append(rec["ms"])
    out = []
    for name, _, _ in arms:
        row = rows[name]
        row.update(ms=round(statistics.median(row["ms_runs"]), 1), ms_min=min(row["ms_runs"]), ms_max=max(row["ms_runs"]))
        out.append(row)
        print(f"{workload:8s} {name:10s} {row['ms']:9.1f} ms ({row['ms_min']:.1f} .. {row['ms_max']:.1f})  mean spp "
              f"{row['mean_spp']:7.1f}  relMSE {row['rel_mse']:.3e}", file=sys.stderr)
    return dict(workload=bench.WORKLOAD_TEXT, spp=spp, repeats=repeats, reference=dict(spp=ref_spp, **ref_rec), arms=out)


def c2_overhead(waves, rounds):
    n_tris = bench.DEFAULT_TRIS["soup"]
    bench.select_workload("soup", n_tris)
    scene = Y.Scene(bench.scene_path(n_tris, "soup"))
    spp = 4 * waves
    cam = Y.make_camera(bench.W, bench.H, bench.CAM["focal"], bench.CAM["fnum"], bench.CAM["pos"], bench.CAM["target"], (0, 0, 0),
                        bench.CAM["exposure"])
    ctxs = {}
    for arm in ("off", "threshold 0"):
        ctx = Y.Context(max_depth=bench.MAX_DEPTH, traversal=Y.TRAVERSAL_AUTO)
        ctx.upload_scene(scene)
        ctx.set_camera(cam)
        ctxs[arm] = ctx

    def frame(arm):
        ctx = ctxs[arm]
        ctx.begin_frame(bench.W, bench.H, spp, 64)
        if arm != "off":
            ctx.set_adaptive(0.0, 0, LUMA_FLOOR)
        t0 = time.perf_counter()
        for k in range(waves):
            ctx.render_wave(4 * k, 4, 4 * k)
        ms = (time.perf_counter() - t0) * 1e3 / waves
        return ms, ctx.resolve(want_ldr=False)[0]

    for arm in ctxs:  # warm-up
        frame(arm)
    times = {arm: [] for arm in ctxs}
    frames = {}
    for r in range(rounds):
        for arm in (list(ctxs) if r % 2 == 0 else list(ctxs)[::-1]):
            ms, frames[arm] = frame(arm)
            times[arm].append(ms)
    identical = bool((frames["off"].view(np.uint32) == frames["threshold 0"].view(np.uint32)).all())
    for ctx in ctxs.values():
        ctx.close()
    med = {arm: statistics.median(v) for arm, v in times.items()}
    out = dict(workload=bench.WORKLOAD_TEXT, waves_per_frame=waves, wave_samples=4, rounds=rounds,
               ms_per_wave={arm: [round(x, 3) for x in v] for arm, v in times.items()},
               median_ms_per_wave={arm: round(v, 3) for arm, v in med.items()},
               overhead_pct=round(100.0 * (med["threshold 0"] / med["off"] - 1.0), 2), frames_identical=identical)
    print(f"C2 per wave: off {med['off']:.3f} ms, threshold 0 {med['threshold 0']:.3f} ms ({out['overhead_pct']:+.2f} %), "
          f"frames identical: {identical}", file=sys.stderr)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--spp", type=int, default=1024)
    ap.add_argument("--ref-spp", type=int, default=4096)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--c2-waves", type=int, default=40)
    ap.add_argument("--c2-rounds", type=int, default=7)
    ap.add_argument("--workloads", default="sponza,mclaren")
    ap.add_argument("--out")
    args = ap.parse_args()
    Y.use_library(Y.capi.load())
    out = dict(gpu_info(), quality=[quality(w, args.spp, args.ref_spp, args.repeats) for w in args.workloads.split(",") if w],
               c2_overhead=c2_overhead(args.c2_waves, args.c2_rounds))
    out.update(gpu_info_after=gpu_info())
    text = json.dumps(out, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
