"""First-hit AOVs (yc_enable_aovs / yr_enable_aovs, include/yart_cuda.h) and PFM output.

1. Oracle: the camera rays of the frame (yc_generate_primary_rays) traced with the matching walk, the base colour read
   from the scene's materials, summed in float32 in sample order by numpy: equal to yc_resolve_aovs bit for bit.
2. The frames and ray counts do not change when AOVs are on, however the work is cut.
3. The AOVs do not change however the work is cut, and the CUDA build equals the CPU build.
4. Renderers over several contexts or processes give the planes of one context.
5. The refusals; 6. the PFM writer.
The CPU part runs the CPU build of the same sources (tests/hostsim); the `-m gpu` part the CUDA library.  Every
context names its traversal."""
import ctypes as C
import os
import socket
import subprocess
import sys
import threading

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:  # run as a script: the worker of the two-process test
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import pytest  # noqa: E402

import harness as H  # noqa: E402
import yart_b200 as Y  # noqa: E402
from yart_b200 import scenes  # noqa: E402

MAT_DT = np.dtype({"names": ["base", "baseTex"], "formats": [("<f4", 3), "<i4"], "offsets": [0, 144], "itemsize": 184})
TRACE_FLAG = {Y.TRAVERSAL_REFERENCE_ORDER: Y.TRACE_REFERENCE_ORDER, Y.TRAVERSAL_AUTO: Y.TRACE_WIDE}
TRAVERSALS = [Y.TRAVERSAL_REFERENCE_ORDER, Y.TRAVERSAL_AUTO]


# ------------------------------------------------------------------------------------------
# scenes
# ------------------------------------------------------------------------------------------
def cached_scene(tag, make):
    path = os.path.join(H.CACHE, f"aov_{tag}.ysc")
    if not os.path.exists(path):
        os.makedirs(H.CACHE, exist_ok=True)
        tmp = path + f".tmp{os.getpid()}"
        make().write(tmp)
        os.replace(tmp, path)
    return path


def modified(s, base_textures=True, alpha=True):
    """Scene `s` without base textures and / or with every texel opaque."""
    for m in s.materials:
        if not base_textures:
            m.base_tex = -1
    for t in s.textures:
        if not alpha and t.data.dtype == np.uint8 and t.data.shape[-1] == 4:
            t.data[..., 3] = 255
    return s


def case(name):
    """Scene file and frame settings: cornell, seedN (randomised: normal maps, nested transforms), mclaren (186 K
    triangles); a suffix _plain drops base textures and alpha, _opaque alpha only."""
    base, _, kind = name.partition("_")
    kw = dict(base_textures=kind == "opaque" or kind == "", alpha=kind == "")
    if base == "cornell":
        cam, w, h, spp, depth = H.scene_camera("cornell"), 48, 40, 16, 30
        path = cached_scene(name, lambda: modified(scenes.cornell(), **kw))
    elif base == "mclaren":
        cam, w, h, spp, depth = H.scene_camera("mclaren"), 96, 54, 4, 12
        path = cached_scene(name, lambda: modified(scenes.mclaren(n_tris=200_000, env_res=64), **kw))
    else:
        seed = int(base[4:])
        cam = scenes.random_scene(seed).camera
        w, h, spp, depth = cam["w"], cam["h"], 16, 30 if seed % 5 else 3
        path = cached_scene(name, lambda: modified(scenes.random_scene(seed), **kw))
    return dict(path=path, cam=cam, w=w, h=h, spp=spp, depth=depth, tile=16)


def camera(c):
    cam = c["cam"]
    return Y.make_camera(c["w"], c["h"], cam["focal"], cam["fnum"], cam["pos"], cam["target"], (0, 0, 0), cam["exposure"],
                         cam.get("sides", 0))


def progressive(spp):
    out, left, ws = [], spp, 1
    while left:
        out.append(min(ws, left))
        left -= out[-1]
        ws *= 2
    return out


# variants that change how a frame's work is cut: context options, wave sizes (None: one wave), waves in flight
VARIANTS = {
    "default": (dict(), None, False),
    "tail_every_bounce": (dict(tail_threshold=1 << 16), None, False),
    "tail_never": (dict(tail_threshold=-1), None, False),
    "small_capacity": (dict(max_paths="small"), None, False),
    "spill_stack": (dict(sh_stack_entries=2), None, False),
    "waves_in_flight": (dict(), "progressive", True),
    "progressive": (dict(), "progressive", False),
}


def render(c, traversal, aovs, variant="default", sc=None, waves=None):
    """(hdr, ldr, counts, aov planes, context, scene): the frame through yc_render_wave[_async] (`waves`: wave sizes)."""
    opts, wv, async_waves = VARIANTS[variant]
    opts = dict(opts)
    if opts.get("max_paths") == "small":
        opts["max_paths"] = c["w"] * c["h"] // 3
    sc = sc or Y.Scene(c["path"])
    ctx = Y.Context(max_depth=c["depth"], traversal=traversal, **opts)
    ctx.upload_scene(sc)
    ctx.set_camera(camera(c))
    if aovs:
        ctx.enable_aovs()
    ctx.begin_frame(c["w"], c["h"], c["spp"], c["tile"], (0.1, 0.2, 0.3), Y.TONEMAP_AGX)
    taken = 0
    for n in waves or (progressive(c["spp"]) if wv == "progressive" else [c["spp"]]):
        (ctx.render_wave_async if async_waves else ctx.render_wave)(taken, n, taken)
        taken += n
    if async_waves:
        ctx.wave_sync()
    hdr, ldr, st = ctx.resolve()
    planes = ctx.resolve_aovs() if aovs else None
    counts = (st.raysReference, st.raysExtend, st.raysShadow, st.samples)
    return hdr, ldr, counts, planes, ctx, sc


# ------------------------------------------------------------------------------------------
# 1. the oracle
# ------------------------------------------------------------------------------------------
def pixel_list(w, h, tile):
    """The frame's pixels in the order of the pixel list (tiles row-major, pixels row-major inside)."""
    xs, ys = [], []
    for ty in range(0, h, tile):
        for tx in range(0, w, tile):
            for y in range(ty, min(ty + tile, h)):
                for x in range(tx, min(tx + tile, w)):
                    xs.append(x), ys.append(y)
    return np.array(xs), np.array(ys)


def oracle(ctx, sc, c, trace_flag, batch=4):
    """The AOV planes of the frame's samples [0, spp), from traced camera rays, in float32 and sample order."""
    w, h = c["w"], c["h"]
    n = w * h
    mats = np.frombuffer((C.c_char * (MAT_DT.itemsize * sc.flat.nMaterials)).from_address(sc.flat.materials), MAT_DT)
    assert (mats["baseTex"] < 0).all(), "the oracle reads YcMaterial::base: scenes without base textures only"
    base = mats["base"].astype(np.float32)
    sum_b, sum_n, sum_t = np.zeros((n, 3), np.float32), np.zeros((n, 3), np.float32), np.zeros(n, np.float32)
    hits_n = np.zeros(n, np.int64)
    for s0 in range(0, c["spp"], batch):
        k = min(batch, c["spp"] - s0)
        dev = ctx.device_alloc(n * k * 32)
        ctx.generate_primary_rays(s0, k, dev)
        rays = np.empty((n * k, 8), np.float32)
        ctx.d2h(rays, dev)
        ctx.device_free(dev)
        hits, _ = ctx.trace(rays, Y.TRACE_CLOSEST | trace_flag)
        for s in range(k):  # sample-major: ray s * n + p is sample s0 + s of pixel p
            hs = hits[s * n:(s + 1) * n]
            m = hs["didHit"] == 1
            sum_b[m] += base[hs["material"][m]]
            sum_n[m] += hs["n"][m]
            sum_t[m] += hs["t"][m]
            hits_n += m
    S, Hc = np.float32(c["spp"]), hits_n.astype(np.float32)
    albedo = np.concatenate([sum_b / S, (Hc / S)[:, None]], 1)
    depth = np.divide(sum_t, Hc, out=np.zeros_like(sum_t), where=hits_n > 0)
    nd = np.concatenate([sum_n / S, depth[:, None]], 1)
    xs, ys = pixel_list(w, h, c["tile"])
    out_a, out_n = np.zeros((h, w, 4), np.float32), np.zeros((h, w, 4), np.float32)
    out_a[ys, xs], out_n[ys, xs] = albedo, nd
    return out_a, out_n

ORACLE_CASES = ["cornell_plain", "seed3_plain", "seed8_plain", "seed27_plain", "seed111_plain", "mclaren_plain"]


def check_oracle(name, traversal):
    c = case(name)
    hdr, ldr, counts, (albedo, nd), ctx, sc = render(c, traversal, aovs=True)
    ref_a, ref_n = oracle(ctx, sc, c, TRACE_FLAG[traversal])
    assert H.bits_equal(albedo, ref_a).all(), f"{name}: albedo differs from the traced oracle"
    assert H.bits_equal(nd, ref_n).all(), f"{name}: normal / depth differs from the traced oracle"
    assert 0 < albedo[..., 3].mean() <= 1 and (nd[..., 3] >= 0).all()
    ctx.close()


@pytest.mark.parametrize("traversal", TRAVERSALS)
@pytest.mark.parametrize("name", ORACLE_CASES)
def test_aovs_equal_traced_oracle_hostsim(name, traversal, hostsim_lib):
    check_oracle(name, traversal)


@pytest.mark.gpu
@pytest.mark.parametrize("traversal", TRAVERSALS)
@pytest.mark.parametrize("name", ORACLE_CASES)
def test_aovs_equal_traced_oracle_cuda(name, traversal, cuda_lib):
    check_oracle(name, traversal)


@pytest.mark.gpu
def test_aovs_equal_traced_oracle_c2_1080p(cuda_lib):
    """C2 as bench.py builds it: the 1 M-triangle soup at 1920x1080, depth 1, one wave of 4 samples."""
    import bench
    bench.select_workload("soup", bench.DEFAULT_TRIS["soup"])
    cam = dict(bench.CAM, sides=0)
    c = dict(path=bench.scene_path(bench.DEFAULT_TRIS["soup"], "soup"), cam=cam, w=bench.W, h=bench.H, spp=4, depth=bench.MAX_DEPTH,
             tile=64)
    hdr, ldr, counts, (albedo, nd), ctx, sc = render(c, Y.TRAVERSAL_AUTO, aovs=True)
    ref_a, ref_n = oracle(ctx, sc, c, Y.TRACE_WIDE, batch=1)
    assert H.bits_equal(albedo, ref_a).all() and H.bits_equal(nd, ref_n).all()
    ctx.close()


# ------------------------------------------------------------------------------------------
# 2. + 3. frames untouched, AOVs invariant, CUDA = CPU
# ------------------------------------------------------------------------------------------
# (scene, traversal): textured + alpha-tested scenes walk the reference-order BVH; opaque textured ones the wide one
BEAUTY_CASES = [("seed8", Y.TRAVERSAL_REFERENCE_ORDER), ("seed27", Y.TRAVERSAL_REFERENCE_ORDER), ("seed8_opaque", Y.TRAVERSAL_AUTO),
                ("seed111_opaque", Y.TRAVERSAL_AUTO), ("cornell", Y.TRAVERSAL_REFERENCE_ORDER), ("cornell", Y.TRAVERSAL_AUTO)]


def check_variants(name, traversal):
    """Every variant: the frames and counts equal the AOV-less default's, the AOVs equal the default's."""
    c = case(name)
    sc = Y.Scene(c["path"])
    planes0 = None
    for v in VARIANTS:
        hdr_off, ldr_off, counts_off, _, ctx, _ = render(c, traversal, aovs=False, variant=v, sc=sc)
        ctx.close()
        hdr, ldr, counts, planes, ctx, _ = render(c, traversal, aovs=True, variant=v, sc=sc)
        ctx.close()
        assert H.bits_equal(hdr, hdr_off).all() and H.bits_equal(ldr, ldr_off).all(), f"{name} {v}: AOVs changed the frame"
        assert counts == counts_off, f"{name} {v}: AOVs changed the ray counts"
        planes0 = planes0 or planes
        assert all(H.bits_equal(a, b).all() for a, b in zip(planes, planes0)), f"{name} {v}: the AOVs depend on how the work is cut"
    return planes0


@pytest.mark.parametrize("name,traversal", BEAUTY_CASES)
def test_aovs_leave_frames_alone_and_do_not_depend_on_the_cut_hostsim(name, traversal, hostsim_lib):
    check_variants(name, traversal)


@pytest.mark.gpu
@pytest.mark.parametrize("name,traversal", BEAUTY_CASES)
def test_aovs_leave_frames_alone_and_do_not_depend_on_the_cut_cuda(name, traversal, cuda_lib):
    planes = check_variants(name, traversal)
    Y.use_library(H.hostsim())
    ref = render(case(name), traversal, aovs=True)
    ref[4].close()
    assert all(H.bits_equal(a, b).all() for a, b in zip(planes, ref[3])), f"{name}: the CUDA build's AOVs differ from the CPU build's"


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["seed3", "seed3_opaque", "seed3_plain", "seed40", "seed40_opaque", "seed40_plain", "mclaren_plain"])
def test_aovs_cuda_equal_cpu_build(name, cuda_lib):
    c = case(name)
    got = render(c, Y.TRAVERSAL_AUTO, aovs=True, variant="progressive")
    got[4].close()
    Y.use_library(H.hostsim())
    ref = render(c, Y.TRAVERSAL_AUTO, aovs=True, variant="progressive")
    ref[4].close()
    assert all(H.bits_equal(a, b).all() for a, b in zip(got[3], ref[3]))
    assert all(H.bits_equal(a, b).all() for a, b in zip(got[:2], ref[:2]))


def check_one_wave_equals_waves_of_1_2_4_8(name, traversal):
    c = case(name)
    one, prog = render(c, traversal, True, waves=[15]), render(c, traversal, True, waves=[1, 2, 4, 8])
    one[4].close(), prog[4].close()
    assert all(H.bits_equal(a, b).all() for a, b in zip(one[3], prog[3]))


@pytest.mark.parametrize("name,traversal", BEAUTY_CASES)
def test_one_wave_equals_waves_of_1_2_4_8_hostsim(name, traversal, hostsim_lib):
    check_one_wave_equals_waves_of_1_2_4_8(name, traversal)


@pytest.mark.gpu
@pytest.mark.parametrize("name,traversal", BEAUTY_CASES)
def test_one_wave_equals_waves_of_1_2_4_8_cuda(name, traversal, cuda_lib):
    check_one_wave_equals_waves_of_1_2_4_8(name, traversal)


# ------------------------------------------------------------------------------------------
# 4. renderers over several contexts / processes
# ------------------------------------------------------------------------------------------
def renderer(c, **kw):
    return Y.Renderer(c["w"], c["h"], camera(c), Y.Scene(c["path"]), samples=c["spp"], first_wave_samples=4, max_wave_samples=8,
                      max_depth=c["depth"], tile_size=c["tile"], traversal=Y.TRAVERSAL_AUTO, aovs=True, **kw)


def check_multi(devices):
    c = case("seed8_opaque")
    r1 = renderer(c)
    r1.render_sync()
    one = r1.read_aovs()
    r1.close()
    rn = renderer(c, devices=devices)
    for _ in range(2):  # the second render starts from cleared sums
        rn.render_sync()
        got = rn.read_aovs()
        for k in one:
            assert H.bits_equal(got[k], one[k]).all(), f"{k} of {len(devices)} contexts differs from one context's"
    rn.close()
    assert set(one) == {"albedo", "coverage", "normal", "depth"} and one["albedo"].shape == (c["h"], c["w"], 3)


def test_in_process_group_equals_one_context_hostsim(hostsim_lib):
    check_multi([0, 0, 0])


@pytest.mark.gpu
def test_in_process_group_equals_one_context_cuda(cuda_lib):
    check_multi([0, 0, 0])


@pytest.mark.gpu
def test_two_gpus_equal_one_context(cuda_lib):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("one GPU")
    check_multi([0, 1])


def free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def dist_worker(rank, world, port, out_dir):
    """One rank of a yr_create_dist_custom renderer over gloo (run as `python test_aovs.py rank world port out_dir`)."""
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

    r = renderer(case("seed8_opaque"), dist=(rank, world, collective))
    r.render_sync()
    got = r.read_aovs()
    if rank == 0:
        np.savez(os.path.join(out_dir, "aovs.npz"), **got)
    r.close()
    dist.barrier()
    dist.destroy_process_group()


def test_two_processes_equal_one_context_hostsim(tmp_path, hostsim_lib):
    H.hostsim()
    case("seed8_opaque")
    port = free_port()
    procs = [subprocess.Popen([sys.executable, __file__, str(r), "2", str(port), str(tmp_path)], stdout=subprocess.PIPE,
                              stderr=subprocess.STDOUT, text=True) for r in range(2)]
    for p in procs:
        out, _ = p.communicate(timeout=300)
        assert p.returncode == 0, out[-3000:]
    r1 = renderer(case("seed8_opaque"))
    r1.render_sync()
    one = r1.read_aovs()
    r1.close()
    got = np.load(tmp_path / "aovs.npz")
    for k in one:
        assert H.bits_equal(got[k], one[k]).all()


# ------------------------------------------------------------------------------------------
# 5. refusals
# ------------------------------------------------------------------------------------------
def expect(rc_name, fn):
    with pytest.raises(Y.YartError, match=f"YC_ERR_{rc_name}"):
        fn()


def check_refusals():
    c = case("cornell")
    naive = Y.Context(integrator=Y.INTEGRATOR_NAIVE, traversal=Y.TRAVERSAL_AUTO)
    expect("UNSUPPORTED", naive.enable_aovs)
    naive.close()
    expect("UNSUPPORTED", lambda: renderer(c, integrator=Y.INTEGRATOR_NAIVE))
    expect("UNSUPPORTED", lambda: renderer(c, devices=[0, 0], sharding=Y.SHARD_BUCKETS))

    sc = Y.Scene(c["path"])
    ctx = Y.Context(max_depth=4, traversal=Y.TRAVERSAL_AUTO)
    ctx.upload_scene(sc)
    ctx.set_camera(camera(c))
    ctx.begin_frame(c["w"], c["h"], 8, 16)
    expect("STATE", ctx.resolve_aovs)  # not enabled
    ctx.enable_aovs()  # before the frame's first wave: allowed
    expect("UNSUPPORTED", lambda: ctx.accumulate_wave(0, 4, 0, 2))
    ctx.render_wave(0, 4, 0)
    expect("STATE", ctx.enable_aovs)  # inside the frame
    expect("STATE", lambda: ctx.enable_aovs(False))
    a, n = ctx.resolve_aovs()
    assert a[..., 3].max() > 0
    ctx.begin_frame(c["w"], c["h"], 8, 16)
    a, n = ctx.resolve_aovs()  # cleared by yc_begin_frame
    assert not a.any() and not n.any()
    ctx.enable_aovs(False)
    expect("STATE", ctx.resolve_aovs)
    expect("STATE", ctx.resolve_aovs_combined)
    ctx.close()

    c = dict(c, w=64, h=64)
    r = Y.Renderer(64, 64, camera(c), Y.Scene(c["path"]), samples=4096, first_wave_samples=8, max_wave_samples=8, max_depth=30,
                   traversal=Y.TRAVERSAL_AUTO)
    expect("STATE", r.read_aovs)  # not enabled
    r.enable_aovs()
    done = threading.Event()
    r.on_done(lambda rd, aborted: done.set())
    r.render()
    assert not done.is_set()
    expect("STATE", r.read_aovs)  # while the render runs
    expect("STATE", lambda: r.enable_aovs(False))
    r.abort()
    r.wait()
    r.read_aovs()
    r.close()


def test_refusals_hostsim(hostsim_lib):
    check_refusals()


@pytest.mark.gpu
def test_refusals_cuda(cuda_lib):
    check_refusals()


# ------------------------------------------------------------------------------------------
# 6. PFM
# ------------------------------------------------------------------------------------------
def read_pfm(path):
    data = open(path, "rb").read()
    magic, dims, scale, rest = data.split(b"\n", 3)
    w, h = (int(v) for v in dims.split())
    ch = {b"PF": 3, b"Pf": 1}[magic]
    assert float(scale) < 0  # little-endian
    a = np.frombuffer(rest, "<f4").reshape(h, w, ch)[::-1]  # stored bottom row first
    return (a if ch == 3 else a[..., 0]), data[:len(magic) + len(dims) + len(scale) + 3]


def test_pfm_round_trip(tmp_path, hostsim_lib):
    rng = np.random.default_rng(5)
    img = rng.standard_normal((5, 7, 4)).astype(np.float32)
    img[0, 0, :] = [-0.0, np.inf, -np.inf, 1e-45]
    p = str(tmp_path / "rgb.pfm")
    Y.write_pfm(p, img[..., :3])
    got, header = read_pfm(p)
    assert header == b"PF\n7 5\n-1.0\n"
    assert (got.view(np.uint32) == img[..., :3].view(np.uint32)).all()
    raw = open(p, "rb").read()[len(header):]
    assert np.frombuffer(raw[:12], "<f4").tobytes() == img[4, 0, :3].tobytes()  # first stored row is the bottom one
    Y.write_pfm(p, img[..., 3])
    got, header = read_pfm(p)
    assert header == b"Pf\n7 5\n-1.0\n" and (got.view(np.uint32) == img[..., 3].view(np.uint32)).all()
    # a channel of strided planes straight from the C entry point: the depth of a normalDepth plane
    rc = Y.lib().ys_write_pfm(p.encode(), img.ctypes.data + 12, 7, 5, 4, 1)
    assert rc == 0
    got, _ = read_pfm(p)
    assert (got.view(np.uint32) == img[..., 3].view(np.uint32)).all()
    assert Y.lib().ys_write_pfm(p.encode(), img.ctypes.data, 7, 5, 4, 2) == Y.capi.YC_ERR_INVALID
    with pytest.raises(ValueError):
        Y.write_pfm(p, img)


if __name__ == "__main__":
    dist_worker(int(sys.argv[1]), int(sys.argv[2]), int(sys.argv[3]), sys.argv[4])
