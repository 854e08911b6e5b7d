#!/usr/bin/env python
"""bench.py — Mrays/s of the render hot path on BASELINE.json configs[1]:
synthetic 1M-triangle random-soup scene, 1920x1080, primary + shadow rays only (maxDepth = 1).

A step = one pass of the hot path over one batch: one wave of SPP samples of every pixel of the
1080p frame (raygen → extend → shade → shadow → accumulate → finalize).

  value      whole-job Mrays/s (reference ray definition, mis-integrator.cpp:22,126) with the scene,
             BVH and camera resident in HBM; timed with CUDA events on the launching stream
  e2e        same metric through the public Renderer API (yr_render_sync + yr_read): per step the
             frame set-up H2D copies and the HDR+LDR frame D2H copies are inside the timed region
  roofline   extend (closest-hit) kernel: algorithmic bytes per launch / its CUDA-event duration
  cpu_baseline  the reference's own tile-threaded CPU renderer (oracle/_ref/oracle_ref_perf) on the
             box's host cores, bounded to 1 spp of the same frame

  parity     the frame of this configuration (1 spp) against the reference's parity build run on this box
  workloads  N = 1: the configs[2] / configs[3] shapes (Sponza- / McLaren-shaped, full MIS+NEE paths) with the
             surface-shading kernel's roofline

N > 1 (torchrun, one rank per GPU): scene replicated; a step is one wave of SPP x N samples of the frame, split over
the ranks by tile (or by GMoN bucket, --sharding buckets) INSIDE libyart_b200.so, which also combines the per-GPU
frames / accumulation buffers with NCCL on its own stream after every wave, inside the timed region (weak scaling:
W*H*SPP camera paths per GPU and step).  `strong` reports the N = 1 step's job split over the N GPUs.  torch.distributed
carries no frame data: barriers, the communicator id and the max-over-ranks of the timings only.
value = rays of all ranks / max-over-ranks device time (CUDA events around every wave and every collective).

--impl reference times the reference CPU renderer alone (all host threads), same metric/config.
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

W, H = 1920, 1080
_REAL_STDOUT = sys.stdout
METRIC = "Mrays/s at 1080p (primary + shadow rays, reference ray count)"


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# workload → (scene generator, kwargs, maxDepth, description).  "soup" is BASELINE.json configs[1] (the bench
# line of record); "sponza" / "mclaren" are configs[2] / configs[3] shapes, full MIS+NEE paths (maxDepth 30).
WORKLOADS = {
    "soup": ("soup", {}, 1, "soup {tris} tris, {W}x{H}, primary+shadow (maxDepth 1)"),
    "sponza": ("sponza", dict(tex_res=512, env_res=1024), 30, "Sponza-shaped {tris} tris, textured PBR + normal maps, HDR env only, {W}x{H}, full paths"),
    "mclaren": ("mclaren", dict(env_res=1024), 30, "McLaren-shaped {tris} tris, clearcoat/chrome/glass+volume, lamps + HDR env, {W}x{H}, full paths"),
}
DEFAULT_TRIS = {"soup": 1_000_000, "sponza": 260_000, "mclaren": 2_000_000}
CAM = dict(pos=(0.0, 0.0, 40.0), target=(0.0, 0.0, 0.0), focal=35.0, fnum=0.0, exposure=0.0)
MAX_DEPTH = 1
WORKLOAD_TEXT = ""


def select_workload(name: str, n_tris: int):
    """Sets the module-level camera / depth / description for the chosen workload."""
    global CAM, MAX_DEPTH, WORKLOAD_TEXT
    from yart_b200 import scenes
    gen, kw, depth, text = WORKLOADS[name]
    small = dict(kw, n_tris=100)
    if "tex_res" in small:
        small["tex_res"] = 4
    if "env_res" in small:
        small["env_res"] = 4
    cam = getattr(scenes, gen)(**small).camera
    CAM = dict(pos=tuple(cam["pos"]), target=tuple(cam["target"]), focal=cam["focal"], fnum=cam["fnum"], exposure=cam["exposure"])
    MAX_DEPTH = depth
    WORKLOAD_TEXT = text.format(tris=n_tris, W=W, H=H)


def scene_path(n_tris: int, workload: str = "soup") -> str:
    import tempfile
    from yart_b200 import scenes
    gen, kw, _, _ = WORKLOADS[workload]
    d = os.environ.get("YART_BENCH_CACHE", os.path.join(tempfile.gettempdir(), "yart_b200_bench"))
    os.makedirs(d, exist_ok=True)
    p = os.path.join(d, f"{gen}_{n_tris}.ysc")
    if not os.path.exists(p):
        t0 = time.time()
        tmp = p + f".tmp{os.getpid()}"
        getattr(scenes, gen)(n_tris=n_tris, **kw).write(tmp)
        os.replace(tmp, p)
        log(f"[bench] generated {p} in {time.time() - t0:.1f}s")
    return p


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 100 ms while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.lines, self.proc = [], None
        if index < 0:
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms",
                                          "200", "-i", str(index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0: float, t1: float) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [l.split(", ") for t, l in self.lines if t0 - 0.05 <= t <= t1 + 0.15] or [l.split(", ") for _, l in self.lines]
        sm, mx, reasons = [], [], set()
        for r in rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.strip().lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def peaks() -> tuple[float, str]:
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def cpu_reference(path: str, steps: int, warmup: int, spp: int = 1) -> dict:
    """The reference's TileRenderer on all host threads: `steps` timed renderSync() calls of
    `spp` samples of the 1080p frame, after `warmup` untimed ones (one process, one BVH build)."""
    exe = os.path.join(ROOT, "oracle", "_ref", "oracle_ref_perf")
    if not os.path.exists(exe):
        exe = os.path.join(ROOT, "oracle", "_ref", "oracle_ref")
    out = "/tmp/yart_bench_ref.bin"
    cmd = [exe, "render", path, out, f"w={W}", f"h={H}", f"spp={spp}", f"maxdepth={MAX_DEPTH}", "tonemap=agx",
           "pos=%g,%g,%g" % CAM["pos"], "target=%g,%g,%g" % CAM["target"], f"focal={CAM['focal']}", f"fnum={CAM['fnum']}",
           f"exposure={CAM['exposure']}", f"repeat={steps + warmup}"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"reference CPU renderer failed: {r.stderr[-2000:]}")
    j = json.loads(r.stdout.strip().splitlines()[-1])
    rays, prev = [], 0
    for tot, ms in j["steps"]:  # m_totalRays accumulates over renderSync calls
        rays.append((tot - prev, ms))
        prev = tot
    timed = rays[warmup:]
    tot_rays, tot_ms = sum(r for r, _ in timed), sum(m for _, m in timed)
    return dict(mrays=tot_rays / tot_ms / 1e3, ms_per_step=tot_ms / len(timed), rays_per_step=tot_rays / len(timed),
                threads=j["threads"], build_ms=j["build_ms"], spp=spp, exe=os.path.basename(exe))


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    path = scene_path(args.tris, args.workload)
    res = cpu_reference(path, args.steps, max(args.warmup, 1), spp=1)
    line = {
        "impl": "reference", "metric": METRIC, "value": res["mrays"], "unit": "Mrays/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": max(args.warmup, 1), "ms_per_step": res["ms_per_step"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD_TEXT, "step": "1 spp of the frame",
                   "bvh_build_ms_excluded": res["build_ms"]},
        "cpu_baseline": {"value": res["mrays"], "unit": "Mrays/s", "cores": res["threads"], "kind": "reference",
                         "sample": f"{args.steps} x 1 spp of the 1080p frame, {res['exe']} (unmodified reference, -O3 -march=x86-64-v3)"},
        "e2e": {"value": res["mrays"], "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "samples_per_s": W * H * 1 / (res["ms_per_step"] / 1e3),
    }
    print(json.dumps(line), file=_REAL_STDOUT, flush=True)


SHADE_BYTES_PER_HIT = 544  # surface shading (ResolveK + SampleK + ShadeNeeK), algorithmic bytes per hit (DESIGN.md §4):
# path state 92 B read + 92 B written, vertex data of the hit triangle 120 B (3 indices + 3 x (normal, tangent, uv)),
# material record 176 B, shadow request 64 B written; the 112 B surface record the three kernels hand each other is the
# implementation's own traffic and is not counted; + 36 B of texel taps (base colour, metallic-roughness, normal map:
# 4 taps each) on textured materials
SHADE_TEXTURE_BYTES = 36


def oracle_frame(path: str, spp: int = 1):
    """One frame from the PARITY build of the unmodified reference (oracle/_ref/oracle_ref: -O2, no FMA contraction —
    the build every parity test compares with; the throughput baseline uses the -O3 -march build, whose contracted
    arithmetic is not bit-identical to it).  Returns (hdr, ldr, rays) or None."""
    import numpy as np
    import struct
    exe = os.path.join(ROOT, "oracle", "_ref", "oracle_ref")
    if not os.path.exists(exe):
        return None
    out = f"/tmp/yart_bench_parity_{os.getpid()}.bin"
    cmd = [exe, "render", path, out, f"w={W}", f"h={H}", f"spp={spp}", f"first={spp}", f"max={spp}", f"maxdepth={MAX_DEPTH}",
           "tonemap=agx", "pos=%.9g,%.9g,%.9g" % CAM["pos"], "target=%.9g,%.9g,%.9g" % CAM["target"], f"focal={CAM['focal']}",
           f"fnum={CAM['fnum']}", f"exposure={CAM['exposure']}"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        return None
    raw = open(out, "rb").read()
    os.unlink(out)
    ww, hh, rays, _, _, _ = struct.unpack_from("<IIQdId", raw, 0)
    off, n = struct.calcsize("<IIQdId"), ww * hh * 4
    hdr = np.frombuffer(raw, np.float32, n, off).reshape(hh, ww, 4)
    ldr = np.frombuffer(raw, np.float32, n, off + 4 * n).reshape(hh, ww, 4)
    return hdr, ldr, rays


def rel_mse(img, ref, eps=1e-2):
    import numpy as np
    a, b = img[..., :3].astype(np.float64), ref[..., :3].astype(np.float64)
    return float(np.mean((a - b) ** 2 / (b * b + eps)))


DUMP_PIXELS = 1 << 20  # 2 x 16 MB of frame samples + 8 MB of indices: under 64 MB at any frame size


def dump_frame(out_dir: str, hdr, ldr):
    """Writes the HDR and LDR frames (RGBA float32) as out_dir/{hdr,ldr}.npy, each (n, 4), at the pixels listed in
    out_dir/pixel_index.npy (float64, row-major pixel numbers): every pixel when the frame has at most DUMP_PIXELS of
    them, otherwise the same seeded sample of DUMP_PIXELS pixels in every run of the same frame size."""
    import numpy as np
    n = hdr.shape[0] * hdr.shape[1]
    idx = np.arange(n) if n <= DUMP_PIXELS else np.sort(np.random.default_rng(0).choice(n, DUMP_PIXELS, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "pixel_index.npy"), idx.astype(np.float64))
    np.save(os.path.join(out_dir, "hdr.npy"), hdr.reshape(n, 4)[idx])
    np.save(os.path.join(out_dir, "ldr.npy"), ldr.reshape(n, 4)[idx])
    log(f"[bench] wrote the frame of the last timed step ({len(idx)} of {n} pixels) to {out_dir}")


def workload_record(Y, name: str, local: int, trav: int, spp: int, steps: int) -> dict:
    """A BASELINE.json configs[2] / configs[3] shape on one GPU: full MIS+NEE paths, `steps` waves of `spp` samples of the
    1080p frame after 3 warm-up waves, device-timed, with the surface-shading kernel's share and roofline.  `wave32`: the
    same with 32-sample waves — the size class at which the configuration's 1024-spp render schedules its waves
    (TileRenderer: 64 first, 128 max): 8 chunks per lane instead of 1, so the per-path tails that end every chunk of deep
    paths overlap the other lane's next chunk instead of ending the wave."""
    global CAM, MAX_DEPTH, WORKLOAD_TEXT
    saved = (CAM, MAX_DEPTH, WORKLOAD_TEXT)
    tris = DEFAULT_TRIS[name]
    select_workload(name, tris)
    try:
        scene = Y.Scene(scene_path(tris, name))
        cam = Y.make_camera(W, H, CAM["focal"], CAM["fnum"], CAM["pos"], CAM["target"], (0, 0, 0), CAM["exposure"])
        ctx = Y.Context(device=local, max_depth=MAX_DEPTH, traversal=trav)
        ctx.upload_scene(scene)
        ctx.set_camera(cam)
        ctx.set_profiling(1)
        ctx.begin_frame(W, H, spp * (steps + 3 + 2), 64, (0, 0, 0), Y.TONEMAP_AGX)
        for k in range(3):
            ctx.render_wave_async(k * spp, spp, k * spp)
        s0 = ctx.stats()  # (waits for the waves in flight)
        for k in range(3, 3 + steps):
            ctx.render_wave_async(k * spp, spp, k * spp)
        s1 = ctx.stats()
        # the shading kernels' own duration: two more waves with one chunk in flight instead of two (profiling bit 3), so
        # that the CUDA events around ResolveK + SampleK + ShadeNeeK do not also span the other lane's traversal kernels
        ctx.set_profiling(1 | 4 | 8)
        p0 = ctx.stats()
        for k in range(3 + steps, 3 + steps + 2):
            ctx.render_wave(k * spp, spp, k * spp)
        p1 = ctx.stats()
        ctx.set_profiling(1)
        big, nbig = 32, 3
        ctx.begin_frame(W, H, big * (nbig + 1), 64, (0, 0, 0), Y.TONEMAP_AGX)
        ctx.render_wave(0, big, 0)
        b0 = ctx.stats()
        for k in range(1, 1 + nbig):
            ctx.render_wave_async(k * big, big, k * big)
        b1 = ctx.stats()
        wave32 = {"spp_per_step": big, "steps": nbig, "ms_per_step": (b1.gpuMs - b0.gpuMs) / nbig,
                  "value": (b1.raysReference - b0.raysReference) / (b1.gpuMs - b0.gpuMs) / 1e3, "unit": "Mrays/s",
                  "samples_per_s": W * H * big / ((b1.gpuMs - b0.gpuMs) / nbig / 1e3)}
        ctx.close()
        ms = (s1.gpuMs - s0.gpuMs) / steps
        rays = s1.raysReference - s0.raysReference
        hits, shade_ms, n_shade = p1.hitsShaded - p0.hitsShaded, p1.shadeMs - p0.shadeMs, p1.shadeLaunches - p0.shadeLaunches
        per_hit = SHADE_BYTES_PER_HIT + (SHADE_TEXTURE_BYTES if name == "sponza" else 0)
        peak, peak_src = peaks()
        achieved = per_hit * hits / (shade_ms / 1e3) / 1e9 if shade_ms > 0 else 0.0
        return {"workload": WORKLOAD_TEXT, "value": rays / (ms * steps) / 1e3, "unit": "Mrays/s", "ms_per_step": ms,
                "samples_per_s": W * H * spp / (ms / 1e3), "steps": steps, "spp_per_step": spp,
                "traversal": "wide" if (trav != Y.TRAVERSAL_REFERENCE_ORDER and name != "sponza") else "reference order (alpha-tested materials)" if name == "sponza" else "reference order",
                "extend_ms_per_step": (s1.extendMs - s0.extendMs) / steps, "shade_surface_ms_per_step": shade_ms / 2,
                "wave32": wave32,
                "shade_roofline": {"bound": "hbm", "kernel": "ResolveK + SampleK + ShadeNeeK", "achieved": achieved, "peak": peak, "unit": "GB/s",
                                   "frac": achieved / peak, "bytes_per_hit": per_hit, "hits_per_step": hits / 2,
                                   "launches_per_step": n_shade / 2, "timed": "2 waves with one chunk in flight (CUDA events around the three launches of every bounce)", "traffic": None, "peak_source": peak_src}}
    finally:
        CAM, MAX_DEPTH, WORKLOAD_TEXT = saved


def run_ours(args):
    import numpy as np
    import yart_b200 as Y
    from yart_b200 import capi

    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    dist = None
    if world > 1:
        # torch.distributed is the CONTROL plane only (barriers, the communicator id, max-over-ranks of the timings);
        # every byte of frame / accumulation-buffer data moves inside libyart_b200.so (yc_comm_*: NCCL on its own stream)
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    if rank == 0:
        path = scene_path(args.tris, args.workload)
    if dist:
        dist.barrier()
    path = scene_path(args.tris, args.workload)

    Y.use_library(capi.load())  # raises if libyart_b200.so is missing: no fallback
    Y.set_build_device(local)   # the SAH BVH of large meshes is built on this rank's GPU
    t0 = time.time()
    scene = Y.Scene(path)
    log(f"[bench r{rank}] scene {scene.n_tris} tris, BVH build + flatten {scene.build_ms:.0f} ms ({scene.device_builds} mesh(es) on "
        f"the GPU; load {time.time() - t0:.1f}s, includes CUDA start-up)")
    cam = Y.make_camera(W, H, CAM["focal"], CAM["fnum"], CAM["pos"], CAM["target"], (0, 0, 0), CAM["exposure"])
    spp = args.spp
    trav = {"auto": Y.TRAVERSAL_AUTO, "reference": Y.TRAVERSAL_REFERENCE_ORDER, "wide": Y.TRAVERSAL_WIDE}[args.traversal]
    buckets = world > 1 and args.sharding == "buckets"

    def new_comm_id():
        """One communicator id per communicator (ncclGetUniqueId on rank 0, handed to the others over the control plane)."""
        if not dist:
            return None
        box = [Y.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        return box[0]

    def sync_all():
        ctx.wave_sync()  # waves left in flight by yc_render_wave_async
        if dist:
            import torch
            torch.cuda.synchronize()
            dist.barrier()
            torch.cuda.synchronize()

    def max_over_ranks(*vals):
        if not dist:
            return list(vals)
        import torch
        t = torch.tensor(vals, device=f"cuda:{local}", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.tolist()

    def sum_over_ranks(*vals):
        if not dist:
            return list(vals)
        import torch
        t = torch.tensor(vals, device=f"cuda:{local}", dtype=torch.float64)
        dist.all_reduce(t)
        return t.tolist()

    # ---- device-resident arm ---------------------------------------------------------------
    ctx = Y.Context(device=local, max_depth=MAX_DEPTH, traversal=trav)
    ctx.upload_scene(scene)
    ctx.set_camera(cam)
    ctx.set_profiling(os.environ.get('YART_BENCH_NO_PROFILE') is None)
    if dist:
        ctx.comm_init_rank(rank, world, new_comm_id())
    n_warm = max(args.warmup, 3)

    def timed_waves(S, steps, warm):
        """`warm` + `steps` waves of S samples of the frame, sharded over the ranks: tiles of the reference's tile
        list (rank r renders tile k when k % N == r; the frames are reduced to rank 0 after every wave) or (GMoN bucket,
        pixel class) units (the accumulation buffers are all-reduced as int32 inside every wave).  Returns the
        device time of the timed steps (CUDA events around the wave and around its collective, max over ranks),
        whole-job reference rays, traced rays, launches, collective ms, host wall ms."""
        total = S * (warm + steps + 3)
        if buckets:
            ctx.begin_frame(W, H, total, 64, (0, 0, 0), Y.TONEMAP_AGX)
        else:
            ctx.begin_frame(W, H, total, 64, (0, 0, 0), Y.TONEMAP_AGX, shard_index=rank, shard_count=world)

        def step(k):
            if buckets:
                ctx.accumulate_wave(k * S, S, bucket_shard=rank, bucket_shard_count=world)
                ctx.comm_allreduce_buckets(S)
                ctx.finalize_wave(S, k * S)
            else:
                # consecutive waves of one progressive frame are left in flight (yc_render_wave_async): the next wave's
                # chunks start while this wave's tails, bucket sums, finalize kernel and — with several GPUs — its
                # barrier still run; sync_all() below waits for all of them inside the timed region
                ctx.render_wave_async(k * S, S, k * S)
                if dist:
                    ctx.comm_reduce_frames_async(0)

        for k in range(warm):
            step(k)
        sync_all()
        s0 = ctx.stats()
        w0 = time.time()
        for k in range(warm, warm + steps):
            step(k)
        sync_all()
        w1 = time.time()
        s1 = ctx.stats()
        dev = (s1.gpuMs - s0.gpuMs) + (s1.commMs - s0.commMs)
        comm_ms = s1.commMs - s0.commMs
        if dist and not buckets:
            # the waves in flight do not time their barrier separately (it is inside gpuMs): three more waves, waited for
            # one at a time, give the collective's own duration (not part of the timed region)
            for k in range(warm + steps, warm + steps + 3):
                ctx.render_wave(k * S, S, k * S)
                ctx.comm_reduce_frames(0)
            comm_ms = (ctx.stats().commMs - s1.commMs) / 3 * steps
        dev, comm, wall = max_over_ranks(dev, comm_ms, (w1 - w0) * 1e3)
        rays, traced, launches = sum_over_ranks(s1.raysReference - s0.raysReference,
                                                (s1.raysExtend - s0.raysExtend) + (s1.raysShadow - s0.raysShadow),
                                                s1.kernelLaunches - s0.kernelLaunches)
        return dict(dev_ms=dev, comm_ms=comm, wall_ms=wall, rays=rays, traced=traced, launches=launches, w0=w0, w1=w1, s0=s0, s1=s1,
                    step=step, total_waves=warm + steps)

    # started before the warm-up: nvidia-smi needs ~0.3 s to print its first sample.  Rank 0 samples its own
    # GPU only: eight concurrent nvidia-smi pollers contend for the driver lock and perturb the step time.
    clocks = ClockSampler(local if rank == 0 else -1)
    S_weak = spp * world  # weak scaling: the wave grows with the GPU count, every GPU keeps W*H*spp camera paths per step
    weak = timed_waves(S_weak, args.steps, n_warm)
    dumped = None
    if args.dump_outputs and rank == 0:
        # the frame as it stands after the last timed wave (the padding steps below render more waves), read on the root
        # as yr_read does (combined tile shards); written once the clock window has closed
        dumped = ctx.resolve_combined() if dist and not buckets else ctx.resolve()[:2]
    # keep the GPU under the same load until a few clock samples exist (not timed); the number of
    # extra steps is agreed across ranks so nothing can hang
    el = weak["w1"] - weak["w0"]
    n_extra = int((0.5 - el) / max(el / args.steps, 1e-4)) + 1 if el < 0.5 else 0
    n_extra = int(max_over_ranks(float(n_extra))[0])
    for _ in range(min(n_extra, 200)):
        weak["step"](weak["total_waves"] - 1)
    sync_all()
    clk = clocks.stop(weak["w0"], time.time())
    if dumped:
        dump_frame(args.dump_outputs, *dumped)
    s0, s1 = weak["s0"], weak["s1"]

    frames_direct = bool(dist and not buckets and ctx.comm_frames_direct())
    strong = None
    if dist:
        # the same job as one GPU's step (one wave of `spp` samples of the frame) split over the ranks
        st = timed_waves(spp, args.steps, n_warm)
        strong = {"value": st["rays"] / st["dev_ms"] / 1e3, "unit": "Mrays/s", "ms_per_step": st["dev_ms"] / args.steps,
                  "collective_ms_per_step": st["comm_ms"] / args.steps,
                  "job": f"one wave of {spp} spp of the {W}x{H} frame per step, split over {world} GPUs"}

    # ---- extend-kernel roofline: algorithmic bytes of the reference traversal on these rays ------
    rspp = min(spp, max(1, (1 << 23) // (W * H)))  # roofline launch: at most 8 Mi primary rays (4 spp at 1080p)
    n_rays = W * H * rspp
    rays_dev, hits_dev = ctx.device_alloc(n_rays * 32), ctx.device_alloc(n_rays * 20)
    ctx.begin_frame(W, H, spp * (n_warm + args.steps), 64, (0, 0, 0), Y.TONEMAP_AGX)
    ctx.generate_primary_rays(n_warm * spp, rspp, rays_dev)  # the first timed wave's rays at N = 1
    one = np.array([[0, 0, 40, 0.001, 0.01, 0.02, -0.99975, np.inf]], np.float32)  # any ordinary ray
    import ctypes as C
    lib, h = Y.lib(), ctx._h

    def count_tests(flags):
        ctx.trace(one, Y.TRACE_CLOSEST | Y.TRACE_COUNT | flags)  # zeroes the work counters
        c0 = ctx.stats()
        ms_c = C.c_float()
        assert lib.yc_trace_device(h, rays_dev, n_rays, Y.TRACE_CLOSEST | Y.TRACE_COUNT | flags, hits_dev, 1, C.byref(ms_c)) == 0
        c1 = ctx.stats()
        return c1.boxTests - c0.boxTests, c1.triTests - c0.triTests

    box, tri = count_tests(Y.TRACE_REFERENCE_ORDER)  # SURVEY 8d: the REFERENCE walk's box / triangle tests define the bytes
    wide_on = trav != Y.TRAVERSAL_REFERENCE_ORDER and args.workload != "sponza"
    wbox, wtri = count_tests(Y.TRACE_WIDE) if wide_on else (None, None)
    trace_ms = ctx.trace_device(rays_dev, n_rays, hits_dev, Y.TRACE_CLOSEST, repeat=3)
    ref_walk_ms = ctx.trace_device(rays_dev, n_rays, hits_dev, Y.TRACE_CLOSEST | Y.TRACE_REFERENCE_ORDER, repeat=3) if wide_on else trace_ms
    ctx.device_free(rays_dev)
    ctx.device_free(hits_dev)
    algo_bytes = n_rays * (32 + 20) + 32 * box + 52 * tri
    peak, peak_src = peaks()
    # The dominant kernel is the persistent closest-hit traversal (extendWideKernel / traceWideKernel: the same
    # traceWidePersistent body; extendKernel / traceKernel for the reference-order walk).  Roofline launch = ONE launch
    # over the step's W*H*spp primary rays, timed alone with CUDA events right here (trace_ms, mean of 3 after the step
    # warm-up), against the algorithmic bytes of the REFERENCE's traversal of the same rays.
    n_ext = max(1, s1.extendLaunches - s0.extendLaunches)
    ext_rays = (s1.raysExtend - s0.raysExtend)
    ext_ms_sum = s1.extendMs - s0.extendMs
    in_step = None
    if MAX_DEPTH == 1 and ext_ms_sum > 0:
        step_bytes = algo_bytes / n_rays * ext_rays
        in_step = {"launches": int(n_ext), "rays_per_launch": ext_rays / n_ext, "avg_launch_ms": ext_ms_sum / n_ext,
                   "lanes_in_flight": 2, "aggregate_gbs": step_bytes / (ext_ms_sum / 2 / 1e3) / 1e9}
    roof_kernel = ("traceWidePersistent<closest> (extendWideKernel / traceWideKernel body: 4-wide quantised BVH)" if wide_on else
                   "tracePersistent<closest> (extendKernel / traceKernel body: reference-order BVH2 walk)") + \
        ", one launch over the step's primary rays, timed alone"
    achieved = algo_bytes / (trace_ms / 1e3) / 1e9 if trace_ms > 0 else 0.0
    traffic = None
    tp = os.path.join(ROOT, "profiles", "extend_traffic.json")
    if os.path.exists(tp):
        tj = json.load(open(tp))
        key = "wide" if wide_on else "reference"
        if key in tj:  # DRAM bytes of one ncu-captured launch, scaled to this launch's ray count
            traffic = tj[key]["dram_bytes_per_launch"] * n_rays / tj[key]["rays_per_launch"]

    # ---- end-to-end arm: public Renderer API, host buffers; at N > 1 ONE image: tile shards reduced to rank 0 inside
    # the timed region, a single host read there ------------------------------------------------------------------
    r = Y.Renderer(W, H, cam, scene, samples=S_weak, first_wave_samples=S_weak, max_wave_samples=S_weak, max_depth=MAX_DEPTH,
                   tonemap=Y.TONEMAP_AGX, device=local, traversal=trav, dist=(rank, world, new_comm_id()) if dist else None,
                   sharding=Y.SHARD_BUCKETS if buckets else Y.SHARD_TILES)
    e2e_rays = 0

    def e2e_step():
        nonlocal e2e_rays
        d = r.render_sync()
        if rank == 0:
            r.read(pinned=True)
        e2e_rays = d["total_rays"]  # whole-job figure on every rank

    for _ in range(2):
        e2e_step()
    sync_all()
    e0 = time.time()
    n_e2e = args.steps
    for _ in range(n_e2e):
        e2e_step()
    sync_all()
    e2e_s = max_over_ranks(time.time() - e0)[0]
    r.close()

    # ---- parity of THIS configuration against the reference run on this box (rank 0, N = 1) ----------------------
    parity = None
    if rank == 0 and world == 1 and not args.no_cpu:
        ref = oracle_frame(path, 1)
        if ref is not None:
            rp = Y.Renderer(W, H, cam, scene, samples=1, first_wave_samples=1, max_wave_samples=1, max_depth=MAX_DEPTH,
                            tonemap=Y.TONEMAP_AGX, device=local, traversal=trav)
            dp = rp.render_sync()
            hdr, ldr, _ = rp.read()
            rp.close()
            eq = (hdr.view(np.uint32) == ref[0].view(np.uint32)) | (np.isnan(hdr) & np.isnan(ref[0]))
            parity = {"against": "oracle/_ref/oracle_ref (unmodified reference, -O2 -ffp-contract=off) rendering 1 spp of the same "
                                 "frame on this box", "relmse_hdr": rel_mse(hdr, ref[0]), "relmse_ldr": rel_mse(ldr, ref[1]),
                      "bits_equal_frac": float(eq.all(-1).mean()), "pixels_differing": int((~eq.all(-1)).sum()),
                      "rays": int(dp["total_rays"]), "rays_reference": int(ref[2]), "rays_equal": int(dp["total_rays"]) == int(ref[2])}

    # ---- first frame from a cold start (SURVEY 8f-2: the SAH build is part of what a user waits for) -----------------
    first_frame = None
    if rank == 0 and world == 1:
        t_h = time.time()
        sc_host = Y.Scene(path, bvh_kind=Y.BVH_SAH_HOST)  # the same tree built on the host cores, for comparison
        host_load_ms, host_build_ms = (time.time() - t_h) * 1e3, sc_host.build_ms
        sc_host.close()
        t_a = time.time()
        sc2 = Y.Scene(path)  # reads the description, builds the reference's SAH BVH (large meshes: on the GPU), flattens it
        t_b = time.time()
        r2 = Y.Renderer(W, H, cam, sc2, samples=spp, first_wave_samples=spp, max_wave_samples=spp, max_depth=MAX_DEPTH,
                        tonemap=Y.TONEMAP_AGX, device=local, traversal=trav)
        r2.render_sync()  # uploads the scene (+ collapses it to the wide layout), renders one wave
        r2.read(pinned=True)
        t_c = time.time()
        r2.close()
        sc2.close()
        first_frame = {"total_ms": (t_c - t_a) * 1e3, "scene_load_and_sah_build_ms": (t_b - t_a) * 1e3, "sah_build_ms": sc2.build_ms,
                       "meshes_built_on_gpu": int(sc2.device_builds),
                       "upload_collapse_render_read_ms": (t_c - t_b) * 1e3,
                       "host_builder": {"scene_load_and_sah_build_ms": host_load_ms, "sah_build_ms": host_build_ms,
                                        "total_ms": host_load_ms + (t_c - t_b) * 1e3},
                       "note": "first frame of the same configuration in a process whose CUDA context exists: .ysc read + the "
                               "reference's SAH BVH (yc_build_bvh_sah on the GPU for the 1 M-triangle mesh: the reference's tree, "
                               "node for node; sah_build_ms includes attribute copies and flattening) then upload + BVH4 collapse "
                               f"+ one wave of {spp} spp + frames to the host; host_builder: the same with the tree built on the "
                               "host cores (multithreaded)"}

    if rank == 0:
        cpu = None
        if world == 1 and not args.no_cpu:
            try:
                cr = cpu_reference(path, 2, 1, spp=1)
                cpu = {"value": cr["mrays"], "unit": "Mrays/s", "cores": cr["threads"], "kind": "reference",
                       "sample": f"2 x 1 spp of the same 1080p frame through the unmodified reference's TileRenderer "
                                 f"({cr['exe']}); BVH build {cr['build_ms']:.0f} ms excluded"}
            except Exception as ex:  # noqa: BLE001
                cpu = {"value": None, "unit": "Mrays/s", "cores": os.cpu_count(), "kind": "reference", "sample": f"failed: {ex}"}
        workloads = None
        if world == 1 and args.workload == "soup" and not args.no_workloads:
            workloads = {}
            for name in ("sponza", "mclaren"):
                try:
                    workloads[name] = workload_record(Y, name, local, trav, spp, args.steps)
                except Exception as ex:  # noqa: BLE001
                    workloads[name] = {"error": str(ex)}
        dev_ms = weak["dev_ms"]
        line = {
            "metric": METRIC, "value": weak["rays"] / dev_ms / 1e3, "unit": "Mrays/s", "n_gpus": world, "steps": args.steps,
            "warmup": n_warm, "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD_TEXT,
                       "step": f"one wave of {S_weak} spp of the frame = {spp} spp per GPU ({W * H * spp} camera paths per GPU)",
                       "traversal": ("4-wide quantised BVH collapsed from the reference's SAH tree (YC_TRAVERSAL_AUTO; same triangles, "
                                     "same triangle arithmetic; `parity` below)" if wide_on else "reference-order BVH2 walk (bit-identical frames)"),
                       "parallelism": "single GPU" if world == 1 else
                                      (f"bucket sharding x{world} inside libyart_b200.so: every wave is split into (GMoN bucket, pixel class) "
                                       "units, rank r takes (b + c) % N == r; scene replicated; ncclAllReduce(int32 sum) of the "
                                       "accumulation buffers per wave, inside the timed region") if buckets else
                                      (f"tile sharding x{world} inside libyart_b200.so: rank r renders tile k of the reference's tile list when "
                                       "k % N == r; scene replicated; " +
                                       ("every rank's finalize kernel stores its finished pixels straight into rank 0's HDR + LDR "
                                        "frames over NVLink (rank 0's allocation mapped into the other processes), one small NCCL "
                                        "all-reduce per wave as the barrier, inside the timed region" if frames_direct else
                                        "ncclReduce of the HDR + LDR frames to rank 0 after every wave, inside the timed region")),
                       "l2": "inputs larger than L2: BVH + 0.8 GB of path state streamed per step exceed the 126 MB L2; no flush"},
            "wall_ms_per_step": weak["wall_ms"] / args.steps,
            "collective_ms_per_step": weak["comm_ms"] / args.steps,
            "frame_delivery": None if not dist or buckets else ("direct peer stores + barrier" if frames_direct else "reduce to rank 0"),
            "traced_mrays_per_s": weak["traced"] / dev_ms / 1e3,
            "samples_per_s": W * H * S_weak / (dev_ms / args.steps / 1e3),
            "gpu_launches": int(weak["launches"]),
            "clocks": clk,
            "e2e": {"value": e2e_rays * n_e2e / e2e_s / 1e6, "unit": "Mrays/s",
                    "h2d_bytes_per_step": 256 * world, "d2h_bytes_per_step": 2 * W * H * 16,
                    "call": "Renderer.render_sync() + Renderer.read(pinned=True) on rank 0 (yr_render_sync + yr_read): camera / frame "
                            "description in, ONE image out — the HDR + LDR frames to page-locked host memory" +
                            ("; the ranks' tile shards are reduced to rank 0 by the library inside the timed region" if dist else "")},
            "metric_note": "value counts rays as the reference does (path segments + unoccluded NEE rays); traced_mrays_per_s counts every ray traced",
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic if args.workload == "soup" else None, "kernel": roof_kernel, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": algo_bytes, "rays_per_launch": n_rays, "avg_launch_ms": trace_ms,
                         "box_tests_per_ray": box / n_rays, "tri_tests_per_ray": tri / n_rays,
                         "wide_box_tests_per_ray": wbox / n_rays if wbox is not None else None,
                         "wide_tri_tests_per_ray": wtri / n_rays if wtri is not None else None,
                         "reference_order_walk_launch_ms": ref_walk_ms,
                         "in_step_extend_launches": in_step,
                         "note": "algorithmic bytes = SURVEY 8d: (32 B ray + 20 B hit) per ray + 32 B per box test + 52 B per triangle "
                                 "test of the REFERENCE's BVH2 traversal of these rays (counting build of the reference-order walk); "
                                 "frac > 1 is possible: those bytes are served by the L1 / L2, where the BVH is resident, and the "
                                 "wide walk fetches 16 B per box — DRAM moves only `traffic` (profiles/README.md)"},
            "cpu_baseline": cpu,
            "parity": parity,
            "first_frame": first_frame,
        }
        if strong:
            line["strong"] = strong
        if workloads:
            line["workloads"] = workloads
        print(json.dumps(line), file=_REAL_STDOUT, flush=True)
    ctx.close()
    if dist:
        dist.barrier()
        dist.destroy_process_group()


def main():
    # Only the JSON line may reach stdout: libraries (NCCL prints its version there) write to fd 1 too,
    # so fd 1 is pointed at stderr for the run and the line goes to the saved descriptor.
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10, help="timed steps of the headline, e2e and workload records (cpu_baseline: 2 reference renders)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="soup", choices=sorted(WORKLOADS))
    ap.add_argument("--tris", type=int, default=0, help="triangle count (default: the workload's BASELINE.json size)")
    ap.add_argument("--spp", type=int, default=4)
    ap.add_argument("--sharding", default="tiles", choices=["tiles", "buckets"],
                    help="N > 1: tiles of the reference's tile list per rank (default) or the samples of one wave split by GMoN bucket")
    ap.add_argument("--no-workloads", action="store_true", help="skip the sponza / mclaren sub-records of the default line")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--traversal", default="auto", choices=["auto", "reference", "wide"],
                    help="YcOptions::traversal: auto = the 4-wide BVH for scenes without alpha-tested materials (default), "
                         "reference = the reference-order BVH2 walk (bit-identical frames)")
    ap.add_argument("--width", type=int, default=1920)
    ap.add_argument("--height", type=int, default=1080, help="3840 x 2160 for the BASELINE.json configs[4] shape")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the frame they produced as DIR/<name>.npy (see dump_frame)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    global W, H, METRIC
    W, H = args.width, args.height
    if (W, H) != (1920, 1080):
        METRIC = METRIC.replace("1080p", f"{W}x{H}")
    if not args.tris:
        args.tris = DEFAULT_TRIS[args.workload]
    select_workload(args.workload, args.tris)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
