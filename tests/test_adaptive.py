"""Adaptive sampling (yc_set_adaptive / yr_set_adaptive, include/yart_cuda.h).

1. Oracle: every sample's exposure-scaled radiance recovered with one-sample Mean waves, the moments, e and the stop rule
   computed by numpy in float32: equal to yc_resolve_adaptive bit for bit, wave after wave.
2. Per-pixel identity: each pixel of an adaptive frame (HDR, LDR, AOVs) equals the frame without adaptive sampling after
   the wave at which its sample count S was reached; S is a cumulative wave size and YcStats.samples = ΣS.
3. Limits: threshold 0 changes nothing; a huge threshold stops every pixel after the first wave and ends the render.
4. The frame, S and e do not depend on how the work is cut (capacity, tail, stack spill, waves in flight, a wave split into
   tile-aligned rectangles, estimator, integrator, a batch of views).
5. Tile sharding over in-process groups (direct delivery) and two processes (summing path): every wave's frame and the
   combined planes equal one context's.
6. The refusals.  7. (GPU) the CUDA build equals the CPU build; check 2 at 1080p on the Sponza- and McLaren-shaped scenes.
The CPU part runs the CPU build of the same sources (tests/hostsim); the `-m gpu` part the CUDA library."""
import os
import subprocess
import sys
import threading

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:  # run as a script: the worker of the two-process test
    sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import numpy as np  # noqa: E402
import pytest  # noqa: E402

import harness as H  # noqa: E402
import test_aovs as A  # noqa: E402  (scene cases, cameras, wave schedules)
import yart_b200 as Y  # noqa: E402

TRAVERSALS = [Y.TRAVERSAL_REFERENCE_ORDER, Y.TRAVERSAL_AUTO]
LUMA_FLOOR = np.float32(1e-3)
_thresholds = {}


# ------------------------------------------------------------------------------------------
# rendering through the device layer
# ------------------------------------------------------------------------------------------
def context(c, traversal, variant="default", **kw):
    opts = dict(A.VARIANTS.get(variant, A.VARIANTS["default"])[0])
    if opts.get("max_paths") == "small":
        opts["max_paths"] = c["w"] * c["h"] // 3
    return Y.Context(max_depth=c["depth"], traversal=traversal, **opts, **kw)


def run(c, traversal, adaptive, variant="default", sc=None, waves=None, aovs=False, estimator=Y.ESTIMATOR_GMON,
        integrator=Y.INTEGRATOR_MIS, cams=None, per_wave=False):
    """One frame through yc_render_wave[_async] in `waves` (default: progressive), adaptive = (threshold, min, floor) or
    None.  Returns dict(hdr, ldr, counts, aovs, samples, error, active (per wave), frames (per wave, if per_wave))."""
    sc = sc or Y.Scene(c["path"])
    ctx = context(c, traversal, variant, integrator=integrator)
    ctx.upload_scene(sc)
    if cams is None:
        ctx.set_camera(A.camera(c))
    else:
        ctx.set_cameras(cams)
    if aovs:
        ctx.enable_aovs()
    ctx.begin_frame(c["w"], c["h"], c["spp"], c["tile"], (0.1, 0.2, 0.3), Y.TONEMAP_AGX, estimator)
    if adaptive is not None:
        ctx.set_adaptive(*adaptive)  # before the frame's first wave
    waves = waves or A.progressive(c["spp"])
    rows = c["h"] * ctx.views
    out = dict(active=[], frames=[], planes=[])
    taken = 0
    for k, n in enumerate(waves):
        if variant == "waves_in_flight":
            ctx.render_wave_async(taken, n, taken)
        elif variant == "rectangles" and k == len(waves) // 2:
            cut = c["tile"]  # tile-aligned: the stop test of each half needs no pixel of the other
            ctx.render_wave(taken, n, taken, rect=(0, 0, c["w"], cut))
            ctx.render_wave(taken, n, taken, rect=(0, cut, c["w"], rows - cut))
        else:
            ctx.render_wave(taken, n, taken)
        taken += n
        if per_wave:
            hdr, ldr, _ = ctx.resolve()
            out["frames"].append((hdr, ldr, ctx.resolve_aovs() if aovs else None))
        if adaptive is not None and variant != "waves_in_flight":
            out["active"].append(ctx.resolve_adaptive()[2])
            if per_wave:
                out["planes"].append(ctx.resolve_adaptive()[:2])
    if variant == "waves_in_flight":
        ctx.wave_sync()
    out["hdr"], out["ldr"], st = ctx.resolve()
    out["counts"] = (st.raysReference, st.raysExtend, st.raysShadow)
    out["stats_samples"] = st.samples
    out["aovs"] = ctx.resolve_aovs() if aovs else None
    if adaptive is not None:
        out["samples"], out["error"], _ = ctx.resolve_adaptive()
    ctx.close()
    return out


def threshold(name, traversal):
    """A threshold that stops some pixels and not others in the middle of the progressive schedule: the median of the
    finite e after the third wave of a run in which nothing stops."""
    key = (name, traversal)
    if key not in _thresholds:
        c = A.case(name)
        r = run(c, traversal, (0.0, 0, float(LUMA_FLOOR)), per_wave=True)
        e = r["planes"][min(2, len(r["planes"]) - 1)][1]
        _thresholds[key] = float(np.median(e[np.isfinite(e)]))
    return _thresholds[key]


def params(name, traversal):
    return (threshold(name, traversal), 3, float(LUMA_FLOOR))


# ------------------------------------------------------------------------------------------
# 1. the oracle
# ------------------------------------------------------------------------------------------
def luma(s):
    return (s[..., 0] * np.float32(0.2126) + s[..., 1] * np.float32(0.7152)) + s[..., 2] * np.float32(0.0722)


def error_of(s1, s2, n, floor):
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        fn = n.astype(np.float32)
        mean = s1 / fn
        var = (s2 - s1 * mean) / (n - 1).astype(np.float32)
        var = np.where(var > 0, var, np.float32(0))
        e = np.sqrt(var / fn) / np.where(mean > floor, mean, floor)
    return np.where(n >= 2, e, np.float32(np.inf)).astype(np.float32)


def stop_rule(e, S, active, tile, thr, min_samples):
    """Pixels of `active` that stop: S >= min_samples and every e of the 3x3 neighbourhood in the tile < thr."""
    h, w = e.shape
    ys, xs = np.mgrid[0:h, 0:w]
    ok = e < np.float32(thr)
    good = np.ones((h, w), bool)
    for dy in (-1, 0, 1):
        for dx in (-1, 0, 1):
            ny, nx = ys + dy, xs + dx
            valid = (ny >= 0) & (ny < h) & (nx >= 0) & (nx < w) & (ny // tile == ys // tile) & (nx // tile == xs // tile)
            good &= ~valid | ok[np.clip(ny, 0, h - 1), np.clip(nx, 0, w - 1)]
    return active & (S >= min_samples) & good


def recovered_samples(c, traversal):
    """(spp, h, w, 3) float32: sample s of every pixel, exposure-scaled, from one-sample Mean waves (takenBefore 0)."""
    sc = Y.Scene(c["path"])
    ctx = context(c, traversal)
    ctx.upload_scene(sc)
    ctx.set_camera(A.camera(c))
    ctx.begin_frame(c["w"], c["h"], c["spp"], c["tile"], (0.1, 0.2, 0.3), Y.TONEMAP_AGX, Y.ESTIMATOR_MEAN)
    out = []
    for s in range(c["spp"]):
        ctx.render_wave(s, 1, 0)
        out.append(ctx.resolve(want_ldr=False)[0][..., :3].copy())
    ctx.close()
    out = np.stack(out)
    assert np.isfinite(out).all(), "the oracle needs finite samples"
    return out


def check_oracle(name, traversal):
    c = A.case(name)
    thr, min_samples, floor = params(name, traversal)
    samples = recovered_samples(c, traversal)
    accepted = (samples >= 0).all(-1)  # GMoN (no sample is NaN)
    Y_ = luma(samples)
    h, w = c["h"], c["w"]
    s1, s2 = np.zeros((h, w), np.float32), np.zeros((h, w), np.float32)
    n, S = np.zeros((h, w), np.int64), np.zeros((h, w), np.int64)
    e = np.full((h, w), np.inf, np.float32)
    active = np.ones((h, w), bool)
    want_active, want_planes, taken = [], [], 0
    for ws in A.progressive(c["spp"]):
        for s in range(taken, taken + ws):
            m = active & accepted[s]
            s1 = np.where(m, s1 + Y_[s], s1).astype(np.float32)
            s2 = np.where(m, s2 + Y_[s] * Y_[s], s2).astype(np.float32)
            n += m
        S += active * ws
        taken += ws
        e = np.where(active, error_of(s1, s2, n, np.float32(floor)), e)
        active &= ~stop_rule(e, S, active, c["tile"], thr, min_samples)
        want_active.append(int(active.sum()))
        want_planes.append((S.copy(), e.copy()))
    got = run(c, traversal, (thr, min_samples, floor), per_wave=True)
    for k, ((S_got, e_got), (S_want, e_want)) in enumerate(zip(got["planes"], want_planes)):
        assert H.bits_equal(e_got, e_want).all(), f"{name} wave {k}: the error plane differs from the numpy oracle"
        assert (S_got == S_want).all(), f"{name} wave {k}: the sample counts differ from the stop rule's"
    assert len(got["planes"]) == len(want_planes) and got["active"] == want_active
    assert 0 < want_active[-1] < h * w, f"{name}: the test wants some pixels stopped and some not ({want_active})"
    return got


ORACLE_CASES = ["cornell", "seed3", "seed8", "seed27", "mclaren"]


@pytest.mark.parametrize("traversal", TRAVERSALS)
@pytest.mark.parametrize("name", ORACLE_CASES)
def test_error_and_stops_equal_numpy_oracle_hostsim(name, traversal, hostsim_lib):
    check_oracle(name, traversal)


@pytest.mark.gpu
@pytest.mark.parametrize("traversal", TRAVERSALS)
@pytest.mark.parametrize("name", ORACLE_CASES)
def test_error_and_stops_equal_numpy_oracle_cuda(name, traversal, cuda_lib):
    check_oracle(name, traversal)


# ------------------------------------------------------------------------------------------
# 2. per-pixel identity with the frames of the render without adaptive sampling
# ------------------------------------------------------------------------------------------
def check_identity(c, traversal, adaptive, waves=None, aovs=True, sc=None):
    waves = waves or A.progressive(c["spp"])
    off = run(c, traversal, None, waves=waves, aovs=aovs, per_wave=True, sc=sc)
    on = run(c, traversal, adaptive, waves=waves, aovs=aovs, sc=sc)
    cum = np.cumsum(waves)
    S = on["samples"]
    assert np.isin(S, cum).all(), "S is not a cumulative wave size"
    assert on["stats_samples"] == int(S.sum())
    wave_of = np.searchsorted(cum, S)
    for k in range(len(waves)):
        m = wave_of == k
        hdr, ldr, planes = off["frames"][k]
        assert H.bits_equal(on["hdr"][m], hdr[m]).all(), f"wave {k}: HDR of the pixels that stopped there differs"
        assert H.bits_equal(on["ldr"][m], ldr[m]).all(), f"wave {k}: LDR of the pixels that stopped there differs"
        if aovs:
            assert all(H.bits_equal(a[m], b[m]).all() for a, b in zip(on["aovs"], planes)), f"wave {k}: AOVs differ"
    return on, off


IDENTITY_CASES = [("cornell", Y.TRAVERSAL_REFERENCE_ORDER), ("cornell", Y.TRAVERSAL_AUTO), ("seed8", Y.TRAVERSAL_REFERENCE_ORDER),
                  ("seed27", Y.TRAVERSAL_AUTO), ("mclaren", Y.TRAVERSAL_AUTO)]


def check_identity_case(name, traversal):
    on, _ = check_identity(A.case(name), traversal, params(name, traversal))
    assert len(set(on["samples"].ravel().tolist())) > 1, "nothing stopped early"


@pytest.mark.parametrize("name,traversal", IDENTITY_CASES)
def test_each_pixel_equals_the_full_render_at_its_last_wave_hostsim(name, traversal, hostsim_lib):
    check_identity_case(name, traversal)


@pytest.mark.gpu
@pytest.mark.parametrize("name,traversal", IDENTITY_CASES)
def test_each_pixel_equals_the_full_render_at_its_last_wave_cuda(name, traversal, cuda_lib):
    check_identity_case(name, traversal)


# ------------------------------------------------------------------------------------------
# 3. limits
# ------------------------------------------------------------------------------------------
def renderer(c, **kw):
    kw.setdefault("first_wave_samples", 4)
    kw.setdefault("max_wave_samples", 8)
    kw.setdefault("traversal", Y.TRAVERSAL_AUTO)
    return Y.Renderer(c["w"], c["h"], A.camera(c), Y.Scene(c["path"]), samples=c["spp"], max_depth=c["depth"], tile_size=c["tile"],
                      **kw)


def check_limits():
    c = A.case("seed8_opaque")
    off = run(c, Y.TRAVERSAL_AUTO, None, aovs=True)
    zero = run(c, Y.TRAVERSAL_AUTO, (0.0, 0, 1e-3), aovs=True)
    assert H.bits_equal(zero["hdr"], off["hdr"]).all() and H.bits_equal(zero["ldr"], off["ldr"]).all()
    assert all(H.bits_equal(a, b).all() for a, b in zip(zero["aovs"], off["aovs"]))
    assert zero["counts"] == off["counts"] and (zero["samples"] == c["spp"]).all()

    # everything stops after the first wave: the renderer runs one wave and completes
    waves = []
    r_off = renderer(c)
    r_off.on_wave_complete(lambda rd, wd: waves.append(wd["rays"]))
    r_off.render_sync()
    r_off.close()
    r = renderer(c, adaptive=(1e30, 4, 1e-3))
    seen, done = [], []
    r.on_wave_complete(lambda rd, wd: seen.append(wd))
    r.on_done(lambda rd, aborted: done.append((rd, aborted)))
    d = r.render_sync()
    assert len(seen) == 1 and done and done[0][1] is False
    assert d["samples_taken"] == 4 and d["total_rays"] == waves[0]
    got = r.read_adaptive()
    assert (got["samples"] == 4).all() and (got["error"] < 1e30).all()
    r.close()


def test_limits_hostsim(hostsim_lib):
    check_limits()


@pytest.mark.gpu
def test_limits_cuda(cuda_lib):
    check_limits()


# ------------------------------------------------------------------------------------------
# 4. invariance to the cut
# ------------------------------------------------------------------------------------------
CUT_VARIANTS = ["tail_every_bounce", "tail_never", "small_capacity", "spill_stack", "waves_in_flight", "rectangles"]
CUT_CASES = [("cornell", Y.TRAVERSAL_REFERENCE_ORDER), ("seed8", Y.TRAVERSAL_REFERENCE_ORDER), ("seed27_opaque", Y.TRAVERSAL_AUTO),
             ("mclaren", Y.TRAVERSAL_AUTO)]


def same(a, b, what):
    for k in ("hdr", "ldr", "error"):
        assert H.bits_equal(a[k], b[k]).all(), f"{what}: {k} differs"
    assert (a["samples"] == b["samples"]).all(), f"{what}: samples differ"
    assert a["counts"] == b["counts"], f"{what}: ray counts differ"
    if a["aovs"] is not None:
        assert all(H.bits_equal(x, y).all() for x, y in zip(a["aovs"], b["aovs"])), f"{what}: AOVs differ"


def check_cut(name, traversal):
    c = A.case(name)
    p = params(name, traversal)
    sc = Y.Scene(c["path"])
    ref = run(c, traversal, p, sc=sc, aovs=True)
    assert len(set(ref["samples"].ravel().tolist())) > 1
    for v in CUT_VARIANTS:
        same(run(c, traversal, p, variant=v, sc=sc, aovs=True), ref, f"{name} {v}")


@pytest.mark.parametrize("name,traversal", CUT_CASES)
def test_the_cut_does_not_matter_hostsim(name, traversal, hostsim_lib):
    check_cut(name, traversal)


@pytest.mark.gpu
@pytest.mark.parametrize("name,traversal", CUT_CASES)
def test_the_cut_does_not_matter_cuda(name, traversal, cuda_lib):
    check_cut(name, traversal)


def check_estimators_and_naive(name, traversal):
    """Per-pixel identity under every estimator and the naive integrator (the moments follow the estimator's accepts)."""
    c = A.case(name)
    p = params(name, traversal)
    for est in (Y.ESTIMATOR_MON, Y.ESTIMATOR_MEAN):
        waves = A.progressive(c["spp"])
        off = run(c, traversal, None, waves=waves, estimator=est, per_wave=True)
        on = run(c, traversal, p, waves=waves, estimator=est)
        wave_of = np.searchsorted(np.cumsum(waves), on["samples"])
        for k in range(len(waves)):
            m = wave_of == k
            assert H.bits_equal(on["hdr"][m], off["frames"][k][0][m]).all(), f"estimator {est} wave {k}"
    c = dict(c, depth=5)
    waves = A.progressive(c["spp"])
    off = run(c, traversal, None, waves=waves, integrator=Y.INTEGRATOR_NAIVE, per_wave=True)
    on = run(c, traversal, p, waves=waves, integrator=Y.INTEGRATOR_NAIVE)
    wave_of = np.searchsorted(np.cumsum(waves), on["samples"])
    for k in range(len(waves)):
        m = wave_of == k
        assert H.bits_equal(on["hdr"][m], off["frames"][k][0][m]).all(), f"naive wave {k}"


@pytest.mark.parametrize("name,traversal", [("cornell", Y.TRAVERSAL_REFERENCE_ORDER), ("seed8_opaque", Y.TRAVERSAL_AUTO)])
def test_estimators_and_naive_integrator_hostsim(name, traversal, hostsim_lib):
    check_estimators_and_naive(name, traversal)


@pytest.mark.gpu
@pytest.mark.parametrize("name,traversal", [("cornell", Y.TRAVERSAL_REFERENCE_ORDER), ("seed8_opaque", Y.TRAVERSAL_AUTO)])
def test_estimators_and_naive_integrator_cuda(name, traversal, cuda_lib):
    check_estimators_and_naive(name, traversal)


def check_views(name, traversal):
    """A batch of 3 views (the case's camera and two moved ones) equals each view rendered alone."""
    c = A.case(name)
    p = params(name, traversal)
    cam = c["cam"]
    cams = []
    for k in range(3):
        pos = tuple(float(v) + 0.05 * k for v in cam["pos"])
        cams.append(Y.make_camera(c["w"], c["h"], cam["focal"], cam["fnum"], pos, cam["target"], (0, 0, 0), cam["exposure"],
                                  cam.get("sides", 0)))
    batch = run(c, traversal, p, cams=cams, aovs=True)
    h = c["h"]
    for k, cm in enumerate(cams):
        one = run(c, traversal, p, cams=[cm], aovs=True)
        rows = slice(k * h, (k + 1) * h)
        for key in ("hdr", "ldr", "error"):
            assert H.bits_equal(batch[key][rows], one[key]).all(), f"view {k}: {key}"
        assert (batch["samples"][rows] == one["samples"]).all()
        assert all(H.bits_equal(a[rows], b).all() for a, b in zip(batch["aovs"], one["aovs"]))


def test_batch_of_views_equals_singles_hostsim(hostsim_lib):
    check_views("seed8", Y.TRAVERSAL_REFERENCE_ORDER)


@pytest.mark.gpu
def test_batch_of_views_equals_singles_cuda(cuda_lib):
    check_views("seed8", Y.TRAVERSAL_REFERENCE_ORDER)


# ------------------------------------------------------------------------------------------
# 5. tile sharding
# ------------------------------------------------------------------------------------------
SHARD_CASE = "seed8_opaque"


def render_waves(r):
    """Render with a frame target; every wave's frame, the last HDR and the planes."""
    c = A.case(SHARD_CASE)
    target = np.zeros((c["h"], c["w"], 4), np.float32)
    frames = []
    r.set_frame_target(target)
    r.on_wave_complete(lambda rd, wd: frames.append(target.copy()))
    r.render_sync()
    hdr = r.read()[0]
    return frames, hdr, r.read_adaptive()


def shard_params():
    return (threshold(SHARD_CASE, Y.TRAVERSAL_AUTO), 4, float(LUMA_FLOOR))


def check_shards(devices):
    c = A.case(SHARD_CASE)
    r1 = renderer(c, adaptive=shard_params())
    one = render_waves(r1)
    r1.close()
    assert len(set(one[2]["samples"].ravel().tolist())) > 1
    rn = renderer(c, devices=devices, adaptive=shard_params())
    for _ in range(2):  # the second render starts from a reset state
        frames, hdr, planes = render_waves(rn)
        assert len(frames) == len(one[0])
        for k, (a, b) in enumerate(zip(frames, one[0])):
            assert H.bits_equal(a, b).all(), f"wave {k}: {len(devices)} contexts differ from one"
        assert H.bits_equal(hdr, one[1]).all()
        assert (planes["samples"] == one[2]["samples"]).all() and H.bits_equal(planes["error"], one[2]["error"]).all()
    rn.close()


@pytest.mark.parametrize("n", [2, 3])
def test_tile_shards_equal_one_context_hostsim(n, hostsim_lib):
    check_shards([0] * n)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [2, 3])
def test_tile_shards_equal_one_context_cuda(n, cuda_lib):
    check_shards([0] * n)


def dist_worker(rank, world, port, out_dir):
    """One rank of a yr_create_dist_custom renderer over gloo (`python test_adaptive.py rank world port out_dir`)."""
    import ctypes as C
    import torch
    import torch.distributed as dist
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    Y.use_library(H.hostsim())
    dt = {0: np.float32, 1: np.int32, 2: np.int64}

    def collective(buf, count, dtype, root):
        arr = np.ctypeslib.as_array(C.cast(buf, C.POINTER(np.ctypeslib.as_ctypes_type(dt[dtype]))), shape=(count,))
        t = torch.from_numpy(arr)
        dist.all_reduce(t) if root < 0 else dist.reduce(t, dst=root)
        return 0

    r = renderer(A.case(SHARD_CASE), dist=(rank, world, collective), adaptive=(float(sys.argv[5]), int(sys.argv[6]), float(sys.argv[7])))
    frames, hdr, planes = render_waves(r)
    if rank == 0:
        np.savez(os.path.join(out_dir, "adaptive.npz"), frames=np.stack(frames), hdr=hdr, **planes)
    r.close()
    dist.barrier()
    dist.destroy_process_group()


def test_two_processes_equal_one_context_hostsim(tmp_path, hostsim_lib):
    p = shard_params()
    r1 = renderer(A.case(SHARD_CASE), adaptive=p)
    frames, hdr, planes = render_waves(r1)
    r1.close()
    port = A.free_port()
    procs = [subprocess.Popen([sys.executable, __file__, str(r), "2", str(port), str(tmp_path)] + [repr(v) for v in p],
                              stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True) for r in range(2)]
    for q in procs:
        out, _ = q.communicate(timeout=300)
        assert q.returncode == 0, out[-3000:]
    got = np.load(tmp_path / "adaptive.npz")
    assert got["frames"].shape[0] == len(frames)
    for k in range(len(frames)):
        assert H.bits_equal(got["frames"][k], frames[k]).all(), f"wave {k}"
    assert H.bits_equal(got["hdr"], hdr).all()
    assert (got["samples"] == planes["samples"]).all() and H.bits_equal(got["error"], planes["error"]).all()


# ------------------------------------------------------------------------------------------
# 6. refusals
# ------------------------------------------------------------------------------------------
def check_refusals():
    c = A.case("cornell")
    expect = A.expect
    sc = Y.Scene(c["path"])
    ctx = Y.Context(max_depth=4, traversal=Y.TRAVERSAL_AUTO)
    ctx.upload_scene(sc)
    ctx.set_camera(A.camera(c))
    for bad in [(-1.0, 0, 1e-3), (float("nan"), 0, 1e-3), (float("inf"), 0, 1e-3), (0.1, 0, 0.0), (0.1, 0, -1.0),
                (0.1, 0, float("inf")), (0.1, 0, float("nan"))]:
        expect("INVALID", lambda: ctx.set_adaptive(*bad))
    ctx.set_adaptive(0.1, 2, 1e-3)  # before the frame: allowed
    ctx.begin_frame(c["w"], c["h"], 8, 16)
    expect("UNSUPPORTED", lambda: ctx.accumulate_wave(0, 4, 0, 2))
    expect("UNSUPPORTED", lambda: ctx.accumulate_wave(0, 4))
    expect("UNSUPPORTED", lambda: ctx.finalize_wave(4, 0))
    ctx.render_wave(0, 4, 0)
    expect("STATE", lambda: ctx.set_adaptive(0.2, 2, 1e-3))  # inside the frame
    expect("STATE", lambda: ctx.set_adaptive(None))
    S, e, active = ctx.resolve_adaptive()
    assert (S == 4).all() and active <= c["w"] * c["h"]
    expect("STATE", ctx.resolve_adaptive_combined)
    ctx.begin_frame(c["w"], c["h"], 8, 16)
    S, e, active = ctx.resolve_adaptive()  # reset by yc_begin_frame
    assert not S.any() and np.isinf(e).all() and active == c["w"] * c["h"]
    ctx.set_adaptive(None)
    expect("STATE", ctx.resolve_adaptive)
    ctx.accumulate_wave(0, 4)  # off again: the split works
    ctx.close()

    expect("UNSUPPORTED", lambda: renderer(c, devices=[0, 0], sharding=Y.SHARD_BUCKETS, adaptive=(0.1, 2, 1e-3)))
    expect("INVALID", lambda: renderer(c, adaptive=(-0.5, 2, 1e-3)))
    c = dict(c, w=64, h=64, spp=4096)
    r = renderer(c, first_wave_samples=8, max_wave_samples=8)
    expect("STATE", r.read_adaptive)  # off
    r.set_adaptive(0.0, 0, 1e-3)
    done = threading.Event()
    r.on_done(lambda rd, aborted: done.set())
    r.render()
    assert not done.is_set()
    expect("STATE", r.read_adaptive)  # while the render runs
    expect("STATE", lambda: r.set_adaptive(None))
    r.abort()
    r.wait()
    r.read_adaptive()
    r.close()


def test_refusals_hostsim(hostsim_lib):
    check_refusals()


@pytest.mark.gpu
def test_refusals_cuda(cuda_lib):
    check_refusals()


# ------------------------------------------------------------------------------------------
# 7. GPU: the CUDA build equals the CPU build; identity at 1080p
# ------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name,traversal", [("seed3", Y.TRAVERSAL_AUTO), ("seed40_opaque", Y.TRAVERSAL_AUTO),
                                            ("mclaren", Y.TRAVERSAL_AUTO), ("seed8", Y.TRAVERSAL_REFERENCE_ORDER)])
def test_cuda_equals_cpu_build(name, traversal, cuda_lib):
    c = A.case(name)
    p = (threshold(name, traversal), 3, float(LUMA_FLOOR))
    got = run(c, traversal, p, aovs=True)
    Y.use_library(H.hostsim())
    same(got, run(c, traversal, p, aovs=True), f"{name}: CUDA vs CPU build")


@pytest.mark.gpu
@pytest.mark.parametrize("workload,traversal", [("sponza", Y.TRAVERSAL_REFERENCE_ORDER), ("mclaren", Y.TRAVERSAL_AUTO)])
def test_identity_1080p(workload, traversal, cuda_lib):
    """Check 2 on the benchmark's Sponza-shaped (alpha-tested, reference-order walk) and McLaren-shaped (wide walk) scenes
    at 1920x1080, 256 samples in waves of 64, 128 and 64."""
    import bench
    bench.select_workload(workload, bench.DEFAULT_TRIS[workload])
    c = dict(path=bench.scene_path(bench.DEFAULT_TRIS[workload], workload), cam=dict(bench.CAM, sides=0), w=bench.W, h=bench.H,
             spp=256, depth=bench.MAX_DEPTH, tile=64)
    sc = Y.Scene(c["path"])
    on, _ = check_identity(c, traversal, (0.05, 64, float(LUMA_FLOOR)), waves=[64, 128, 64], aovs=False, sc=sc)
    assert len(set(on["samples"].ravel().tolist())) > 1


if __name__ == "__main__":
    dist_worker(int(sys.argv[1]), int(sys.argv[2]), int(sys.argv[3]), sys.argv[4])
