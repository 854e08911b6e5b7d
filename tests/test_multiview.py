"""Several camera views in one frame (yc_set_cameras / yr_set_cameras, include/yart_cuda.h).

The sampler depends on the view-local pixel, the sample index and the frame's totalSamples / tileSize only, so every view
of a batch must equal, bit for bit, the frame a context renders for that camera alone: HDR, LDR, AOV planes, and the
batch's ray count is the sum of the singles'.
1. Batch = singles over scenes, view counts, walks, estimators and the naive integrator.
2. The same bits however the work is cut (chunks straddling views, tails, waves in flight, progressive waves,
   rectangles across view boundaries).
3. Sharded renderers (in-process groups, tiles and buckets; two processes over gloo) equal one context's batch.
4. The renderer layer (tile callback, frame target, PPM, Python shapes) and the primary rays of each view.
5. The refusals.
The CPU part runs the CPU build of the same sources (tests/hostsim); the `-m gpu` part the CUDA library.  Every context
names its traversal."""
import os
import socket
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:  # run as a script: the worker of the two-process test
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import pytest  # noqa: E402

import harness as H  # noqa: E402
import yart_b200 as Y  # noqa: E402
from yart_b200 import scenes  # noqa: E402

REF, AUTO = Y.TRAVERSAL_REFERENCE_ORDER, Y.TRAVERSAL_AUTO


# ------------------------------------------------------------------------------------------
# scenes and cameras
# ------------------------------------------------------------------------------------------
def cached_scene(tag, make):
    path = os.path.join(H.CACHE, f"mv_{tag}.ysc")
    if not os.path.exists(path):
        tmp = path + f".tmp{os.getpid()}"
        make().write(tmp)
        os.replace(tmp, path)
    return path


def case(name):
    """Scene file and frame settings: cornell, seedN (random_scene: normal maps, nested transforms, alpha textures),
    mclaren (a small McLaren-shaped scene), soup / mclaren_full (bench.py's C2 and McLaren workloads, GPU only)."""
    if name == "cornell":
        return dict(path=H.scene_file("cornell"), cam=H.scene_camera("cornell"), w=24, h=20, spp=8, depth=30, tile=8)
    if name == "mclaren":
        return dict(path=cached_scene("mclaren", lambda: scenes.mclaren(n_tris=20_000, env_res=32)), cam=H.scene_camera("mclaren"),
                    w=32, h=18, spp=4, depth=12, tile=8)
    if name in ("soup", "mclaren_full"):
        import bench
        wl = "soup" if name == "soup" else "mclaren"
        bench.select_workload(wl, bench.DEFAULT_TRIS[wl])
        return dict(path=bench.scene_path(bench.DEFAULT_TRIS[wl], wl), cam=dict(bench.CAM), w=480, h=270, spp=4,
                    depth=bench.MAX_DEPTH, tile=64)
    seed = int(name[4:])
    cam = scenes.random_scene(seed).camera
    return dict(path=cached_scene(name, lambda: scenes.random_scene(seed)), cam=cam, w=min(cam["w"], 24), h=min(cam["h"], 20),
                spp=8, depth=30 if seed % 5 else 3, tile=8)


def cameras(c, n):
    """n cameras around the case's own: positions, focal lengths, f-numbers (pinhole, disk, 5-sided aperture) and
    exposures (-1 ... +1) all differ."""
    cam = c["cam"]
    pos, target = np.asarray(cam["pos"], np.float64), np.asarray(cam["target"], np.float64)
    dist = float(np.linalg.norm(pos - target)) or 1.0
    out = []
    for v in range(n):
        offset = 0.04 * dist * np.array([v - n / 2, 0.5 * (v % 2), 0.1 * v])
        fnum, sides = [(0.0, 0), (2.8, 0), (4.0, 5)][v % 3]
        exposure = -1.0 + 2.0 * v / (n - 1) if n > 1 else cam["exposure"]
        out.append(Y.make_camera(c["w"], c["h"], cam["focal"] * (1 + 0.15 * v), fnum, tuple(pos + offset), cam["target"], (0, 0, 0),
                                 exposure, sides))
    return out


def progressive(spp):
    out, left, ws = [], spp, 1
    while left:
        out.append(min(ws, left))
        left -= out[-1]
        ws *= 2
    return out


# ------------------------------------------------------------------------------------------
# rendering through the device layer
# ------------------------------------------------------------------------------------------
def context(c, traversal, integrator=Y.INTEGRATOR_MIS, **opts):
    return Y.Context(max_depth=c["depth"], traversal=traversal, integrator=integrator, **opts)


def render(c, cams, traversal, aovs=True, estimator=Y.ESTIMATOR_GMON, integrator=Y.INTEGRATOR_MIS, opts=None, waves=None,
           in_flight=False, rects=None, sc=None):
    """(hdr, ldr, albedo, normalDepth, raysReference) of one frame of len(cams) views, each (V, h, w, 4)."""
    sc = sc or Y.Scene(c["path"])
    ctx = context(c, traversal, integrator, **(opts or {}))
    ctx.upload_scene(sc)
    ctx.set_cameras(cams)
    if aovs:
        ctx.enable_aovs()
    ctx.begin_frame(c["w"], c["h"], c["spp"], c["tile"], (0.1, 0.2, 0.3), Y.TONEMAP_AGX, estimator)
    taken = 0
    for n in waves or [c["spp"]]:
        for rect in rects or [None]:
            (ctx.render_wave_async if in_flight else ctx.render_wave)(taken, n, taken, rect)
        taken += n
    if in_flight:
        ctx.wave_sync()
    hdr, ldr, st = ctx.resolve()
    al, nd = ctx.resolve_aovs() if aovs else (np.zeros_like(hdr), np.zeros_like(hdr))
    ctx.close()
    shape = (len(cams), c["h"], c["w"], 4)
    return hdr.reshape(shape), ldr.reshape(shape), al.reshape(shape), nd.reshape(shape), st.raysReference


def singles(c, cams, traversal, **kw):
    """The views rendered one camera per context, stacked as a batch is."""
    sc = Y.Scene(c["path"])
    parts = [render(c, [cam], traversal, sc=sc, **kw) for cam in cams]
    return tuple(np.concatenate([p[k] for p in parts]) for k in range(4)) + (sum(p[4] for p in parts),)


def assert_same(got, ref, what):
    names = ["hdr", "ldr", "albedo", "normalDepth"]
    for k in range(4):
        for v in range(got[k].shape[0]):
            assert H.bits_equal(got[k][v], ref[k][v]).all(), f"{what}: view {v} {names[k]} differs"
    assert got[4] == ref[4], f"{what}: raysReference {got[4]} != {ref[4]}"


# ------------------------------------------------------------------------------------------
# 1. batch = singles
# ------------------------------------------------------------------------------------------
SCENES = ["cornell", "seed3", "seed8", "seed27", "mclaren"]


def check_batch(name, n, traversal, **kw):
    c = case(name)
    cams = cameras(c, n)
    assert_same(render(c, cams, traversal, **kw), singles(c, cams, traversal, **kw), f"{name} V={n}")


@pytest.mark.parametrize("n", [1, 3, 5])
@pytest.mark.parametrize("name", SCENES)
def test_batch_equals_singles_hostsim(name, n, hostsim_lib):
    check_batch(name, n, REF)


@pytest.mark.parametrize("name", ["cornell", "mclaren"])
def test_batch_equals_singles_wide_walk_hostsim(name, hostsim_lib):
    check_batch(name, 3, AUTO)


@pytest.mark.parametrize("estimator", [Y.ESTIMATOR_MON, Y.ESTIMATOR_MEAN])
def test_batch_equals_singles_estimators_hostsim(estimator, hostsim_lib):
    check_batch("seed8", 3, REF, estimator=estimator)


def test_batch_equals_singles_naive_integrator_hostsim(hostsim_lib):
    check_batch("cornell", 3, REF, aovs=False, integrator=Y.INTEGRATOR_NAIVE)


# ------------------------------------------------------------------------------------------
# 2. the same bits however the work is cut
# ------------------------------------------------------------------------------------------
def cuts(c, n):
    rows = n * c["h"]
    return {
        "small_capacity": dict(opts=dict(max_paths=c["w"] * c["h"] // 2)),  # chunks straddle views
        "tail_every_bounce": dict(opts=dict(tail_threshold=1 << 16)),
        "tail_never": dict(opts=dict(tail_threshold=-1)),
        "waves_in_flight": dict(waves=progressive(c["spp"]), in_flight=True),
        "progressive": dict(waves=progressive(c["spp"])),
        # rectangles across view boundaries, each with its own accumulate and finalize
        "rects": dict(waves=[2, c["spp"] - 2], rects=[(0, 0, c["w"], c["h"] + c["h"] // 2),
                                                      (0, c["h"] + c["h"] // 2, c["w"] // 2, rows - c["h"] - c["h"] // 2),
                                                      (c["w"] // 2, c["h"] + c["h"] // 2, c["w"] - c["w"] // 2,
                                                       rows - c["h"] - c["h"] // 2)]),
    }


def check_cuts(name, traversal, only=None):
    c = case(name)
    cams = cameras(c, 3)
    sc = Y.Scene(c["path"])
    refs = {}  # singles per wave schedule
    for cut, kw in cuts(c, 3).items():
        if only and cut not in only:
            continue
        waves = tuple(kw.get("waves", [c["spp"]]))
        if waves not in refs:
            refs[waves] = singles(c, cams, traversal, waves=list(waves))
        assert_same(render(c, cams, traversal, sc=sc, **kw), refs[waves], f"{name} {cut}")


@pytest.mark.parametrize("name,traversal", [("seed8", REF), ("cornell", AUTO)])
def test_batch_does_not_depend_on_the_cut_hostsim(name, traversal, hostsim_lib):
    check_cuts(name, traversal)


# ------------------------------------------------------------------------------------------
# 3. sharding
# ------------------------------------------------------------------------------------------
def renderer(c, cams, **kw):
    return Y.Renderer(c["w"], c["h"], cams, Y.Scene(c["path"]), samples=c["spp"], first_wave_samples=2, max_wave_samples=4,
                      max_depth=c["depth"], tile_size=c["tile"], background=(0.1, 0.2, 0.3), traversal=AUTO, **kw)


def read_all(r):
    hdr, ldr, st = r.read()
    return hdr, ldr, st.raysReference


def check_sharded(devices, sharding):
    c = case("cornell")
    cams = cameras(c, 3)
    one = renderer(c, cams)
    one.render_sync()
    ref = read_all(one)
    one.close()
    rn = renderer(c, cams, devices=devices, sharding=sharding)
    rn.render_sync()
    got = read_all(rn)
    rn.close()
    assert got[0].shape == (3, c["h"], c["w"], 4)
    assert H.bits_equal(got[0], ref[0]).all() and H.bits_equal(got[1], ref[1]).all() and got[2] == ref[2]


@pytest.mark.parametrize("sharding", [Y.SHARD_TILES, Y.SHARD_BUCKETS])
@pytest.mark.parametrize("devices", [[0, 0], [0, 0, 0]])
def test_in_process_group_equals_one_context_hostsim(devices, sharding, hostsim_lib):
    check_sharded(devices, sharding)


def free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def dist_worker(rank, world, port, out_dir):
    """One rank of a yr_create_dist_custom renderer over gloo (run as `python test_multiview.py rank world port out_dir`)."""
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

    c = case("cornell")
    r = renderer(c, cameras(c, 3), dist=(rank, world, collective))
    r.render_sync()
    hdr, ldr, rays = read_all(r)
    if rank == 0:
        np.savez(os.path.join(out_dir, "frames.npz"), hdr=hdr, ldr=ldr)
    r.close()
    dist.barrier()
    dist.destroy_process_group()


def test_two_processes_equal_one_context_hostsim(tmp_path, hostsim_lib):
    H.hostsim()
    c = case("cornell")
    port = free_port()
    procs = [subprocess.Popen([sys.executable, __file__, str(r), "2", str(port), str(tmp_path)], stdout=subprocess.PIPE,
                              stderr=subprocess.STDOUT, text=True) for r in range(2)]
    for p in procs:
        out, _ = p.communicate(timeout=300)
        assert p.returncode == 0, out[-3000:]
    one = renderer(c, cameras(c, 3))
    one.render_sync()
    hdr, ldr, _ = read_all(one)
    one.close()
    got = np.load(tmp_path / "frames.npz")
    assert H.bits_equal(got["hdr"], hdr).all() and H.bits_equal(got["ldr"], ldr).all()


# ------------------------------------------------------------------------------------------
# 4. the renderer layer and the primary rays
# ------------------------------------------------------------------------------------------
def read_ppm(path):
    data = open(path, "rb").read()
    magic, dims, maxval, rest = data.split(b"\n", 3)
    w, h = (int(v) for v in dims.split())
    return magic, w, h, np.frombuffer(rest, np.uint8)


def test_renderer_layer_hostsim(tmp_path, hostsim_lib):
    c = case("cornell")
    cams = cameras(c, 3)
    tiles_per_view = -(-c["w"] // c["tile"]) * -(-c["h"] // c["tile"])
    ref = singles(c, cams, AUTO, aovs=False, waves=[2, 4, 2])  # the renderer's schedule: 2, 4, then what is left

    r = renderer(c, cams)
    target = np.zeros((3, c["h"], c["w"], 4), np.float32)
    r.set_frame_target(target)
    seen = []
    r.on_tile_complete(lambda rd, t: seen.append((rd["samples_taken"], t["index"], t["total"], t["x"], t["y"], t["w"], t["h"])))
    r.render_sync()
    hdr, ldr, st = r.read()
    assert hdr.shape == ldr.shape == (3, c["h"], c["w"], 4)
    assert H.bits_equal(hdr, ref[0]).all() and H.bits_equal(ldr, ref[1]).all() and st.raysReference == ref[4]
    assert H.bits_equal(target, ldr).all()  # the frame target holds the stacked frame
    # every tile of every view once per wave, in stacked coordinates
    waves = sorted({s for s, *_ in seen})
    assert len(waves) == 3
    for s in waves:
        tiles = [t for t in seen if t[0] == s]
        assert [t[1] for t in tiles] == list(range(3 * tiles_per_view)) and {t[2] for t in tiles} == {3 * tiles_per_view}
        cover = np.zeros((3 * c["h"], c["w"]), np.int32)
        for _, _, _, x, y, w, h in tiles:
            cover[y:y + h, x:x + w] += 1
        assert (cover == 1).all()
    # the PPM is the stacked frame, width x (3 * height)
    p = str(tmp_path / "views.ppm")
    r.write_ppm(p)
    magic, w, h, px = read_ppm(p)
    assert (magic, w, h) == (b"P6", c["w"], 3 * c["h"]) and px.size == 3 * w * h
    Y.write_ppm(str(tmp_path / "ref.ppm"), ldr.reshape(3 * c["h"], c["w"], 4))
    assert open(p, "rb").read() == open(tmp_path / "ref.ppm", "rb").read()
    # a sequence of one camera keeps the view axis; a camera given as such does not
    r.set_camera(cams[:1])
    r.set_frame_target(np.zeros((1, c["h"], c["w"], 4), np.float32))
    r.render_sync()
    assert r.read()[0].shape == (1, c["h"], c["w"], 4)
    r.set_frame_target(None)
    r.set_camera(cams[1])
    r.render_sync()
    hdr1 = r.read()[0]
    assert hdr1.shape == (c["h"], c["w"], 4) and H.bits_equal(hdr1, ref[0][1]).all()
    r.close()


def test_primary_rays_of_each_view_hostsim(hostsim_lib):
    c = case("seed3")
    cams = cameras(c, 3)
    sc = Y.Scene(c["path"])

    def rays(cam_list, spp=2):
        ctx = context(c, REF)
        ctx.upload_scene(sc)
        ctx.set_cameras(cam_list)
        ctx.begin_frame(c["w"], c["h"], c["spp"], c["tile"])
        n = len(cam_list) * c["w"] * c["h"] * spp
        dev = ctx.device_alloc(n * 32)
        ctx.generate_primary_rays(1, spp, dev)
        out = np.empty((spp, len(cam_list), c["w"] * c["h"], 8), np.float32)  # sample-major, then view after view
        ctx.d2h(out, dev)
        ctx.device_free(dev)
        ctx.close()
        return out

    batch = rays(cams)
    for v, cam in enumerate(cams):
        assert H.bits_equal(batch[:, v], rays([cam])[:, 0]).all(), f"view {v}"


# ------------------------------------------------------------------------------------------
# 5. refusals
# ------------------------------------------------------------------------------------------
def expect(rc_name, fn):
    with pytest.raises(Y.YartError, match=f"YC_ERR_{rc_name}"):
        fn()


def check_refusals():
    c = case("cornell")
    cams = cameras(c, 3)
    sc = Y.Scene(c["path"])
    ctx = context(c, AUTO)
    ctx.upload_scene(sc)
    lib = Y.lib()
    arr = (Y.capi.YcCamera * 1)(cams[0])
    assert lib.yc_set_cameras(ctx._h, arr, 0) == Y.capi.YC_ERR_INVALID
    assert lib.yc_set_cameras(ctx._h, None, 1) == Y.capi.YC_ERR_INVALID
    assert lib.yc_set_cameras(ctx._h, arr, 65536) == Y.capi.YC_ERR_INVALID
    ctx.set_cameras(cams)
    ctx.begin_frame(c["w"], c["h"], 4, c["tile"])
    ctx.set_cameras(cams[::-1])  # the same count: allowed, the next wave uses them
    ctx.render_wave(0, 1, 0)
    expect("INVALID", lambda: ctx.render_wave(1, 1, 1, (0, 0, c["w"], 3 * c["h"] + 1)))  # outside the stacked frame
    expect("INVALID", lambda: ctx.render_wave(1, 1, 1, (1, 0, c["w"], c["h"])))
    ctx.set_cameras(cams[:2])  # another count: every wave call is refused until the next begin_frame
    expect("STATE", lambda: ctx.render_wave(1, 1, 1))
    expect("STATE", lambda: ctx.render_wave_async(1, 1, 1))
    expect("STATE", lambda: ctx.accumulate_wave(1, 1))
    expect("STATE", lambda: ctx.finalize_wave(1, 1))
    dev = ctx.device_alloc(3 * c["w"] * c["h"] * 32)
    expect("STATE", lambda: ctx.generate_primary_rays(0, 1, dev))
    ctx.device_free(dev)
    ctx.begin_frame(c["w"], c["h"], 4, c["tile"])
    ctx.render_wave(0, 4, 0)
    assert ctx.resolve()[0].shape == (2 * c["h"], c["w"], 4)
    ctx.close()
    r = renderer(c, cams)
    assert lib.yr_set_cameras(r._h, arr, 0) == Y.capi.YC_ERR_INVALID
    assert lib.yr_set_cameras(r._h, None, 1) == Y.capi.YC_ERR_INVALID
    assert lib.yr_set_cameras(r._h, arr, 65536) == Y.capi.YC_ERR_INVALID
    r.close()


def test_refusals_hostsim(hostsim_lib):
    check_refusals()


# ------------------------------------------------------------------------------------------
# 6.-8. the CUDA library
# ------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_refusals_cuda(cuda_lib):
    check_refusals()


@pytest.mark.gpu
@pytest.mark.parametrize("name,n,traversal", [("seed8", 3, REF), ("seed27", 5, REF), ("mclaren", 3, AUTO), ("cornell", 5, AUTO)])
def test_batch_equals_singles_cuda(name, n, traversal, cuda_lib):
    check_batch(name, n, traversal)


@pytest.mark.gpu
def test_batch_equals_singles_naive_integrator_cuda(cuda_lib):
    check_batch("cornell", 3, REF, aovs=False, integrator=Y.INTEGRATOR_NAIVE)


@pytest.mark.gpu
@pytest.mark.parametrize("name,traversal", [("seed8", REF), ("cornell", AUTO)])
def test_batch_does_not_depend_on_the_cut_cuda(name, traversal, cuda_lib):
    check_cuts(name, traversal)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["mclaren", "seed3"])
def test_cuda_batch_equals_cpu_batch_wide_walk(name, cuda_lib):
    c = case(name)
    cams = cameras(c, 3)
    got = render(c, cams, AUTO, waves=progressive(c["spp"]))
    Y.use_library(H.hostsim())
    assert_same(got, render(c, cams, AUTO, waves=progressive(c["spp"])), f"{name}: CUDA batch vs CPU batch")


@pytest.mark.gpu
@pytest.mark.parametrize("traversal", [REF, AUTO])
@pytest.mark.parametrize("name", ["soup", "mclaren_full"])
def test_sixteen_views_full_size_cuda(name, traversal, cuda_lib):
    """16 views of 480x270 at 4 spp of bench.py's C2 soup and McLaren-shaped scene."""
    check_batch(name, 16, traversal, aovs=False)


@pytest.mark.gpu
def test_two_gpus_tile_sharded_batch_equals_one_gpu(cuda_lib):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("one GPU")
    check_sharded([0, 1], Y.SHARD_TILES)


if __name__ == "__main__":
    dist_worker(int(sys.argv[1]), int(sys.argv[2]), int(sys.argv[3]), sys.argv[4])
