"""The library's default render path, TRAVERSAL_AUTO, which runs the quantised 4-wide walk (csrc/wide_bvh.cuh) on every
scene without alpha-tested materials, held to two references that do not depend on tolerances.

Part A (frames): the CPU build of the same sources (tests/hostsim; serial kernels, tail included) renders each scene
once under AUTO, and that frame is the reference.  The CUDA library must reproduce HDR, LDR and the three ray counts bit
for bit in every configuration that changes how the work is cut: tail hand-over at every bounce or never, small
wavefront capacities (many chunks per wave), the global-memory spill of the traversal stack, waves left in flight,
tile shards, estimator-bucket shards and renderers over 2 or 3 contexts.  The reference-order walk must agree between
the two builds as well.  Scenes: the randomised scenes of test_fuzz_parity with every texel made opaque (all 54 then
run the wide walk; most have thin transmissive materials, so NEE transparency is on the path), the scenes of the wide
goldens without alpha, and a 186 K-triangle McLaren-shaped scene at depth 12 (tails and many chunks).

Part B (NEE transparency): stacks of thin transmissive panes with opaque walls and occluders, traced as any-hit rays.
A float64 reference decides occlusion and forms the product of |n·d|·base over the panes the ray crosses; both walks
must match it, and the CUDA records must equal the CPU build's byte for byte.

The CPU part runs the CPU build alone; the `-m gpu` part compares the CUDA kernels (extendKernel, shadowKernel and
traceKernel over WideWalk, tailKernel<false, WideWalk>) with it.  Every context names its traversal."""
import functools
import itertools
import operator
import os

import numpy as np
import pytest

import harness as H
import parity_common as PC
import yart_b200 as Y
from yart_b200 import scenes
from test_fuzz_parity import TM, case_settings
from test_renderer_gpu import devices
from test_wide_bvh import WIDE_RENDER
from test_wide_bvh_robustness import wide_active

U = 2.0 ** -24  # float32 unit roundoff
KTMIN = 0.001   # kTMin (traverse.cuh): testTriangle accepts kTMin < t < hit.t

# ------------------------------------------------------------------------------------------
# Part A: scenes and frames
# ------------------------------------------------------------------------------------------
FUZZ_SEEDS = (*range(40), *range(100, 114))
CASES = [f"seed{s}" for s in FUZZ_SEEDS] + list(WIDE_RENDER) + ["mclaren_200k"]
# the full configuration matrix: randomised scenes with 3-4 thin transmissive materials and 30-bounce paths (one wave,
# and progressive waves of 1, 1, 2, 4 (, 8) samples), the Cornell box in progressive waves, and the deep McLaren scene
FULL = ["seed8", "seed27", "seed111", "render_cornell_waves.npz", "mclaren_200k"]


def opaque_fuzz_scene(seed):
    """random_scene(seed) with every texel's alpha set to 255: no material is alpha-tested any more."""
    path = os.path.join(H.CACHE, f"random_scene_opaque_seed{seed}.ysc")
    if not os.path.exists(path):
        s = scenes.random_scene(seed)
        for t in s.textures:
            if t.data.dtype == np.uint8 and t.data.shape[-1] == 4:
                t.data[..., 3] = 255
        tmp = path + f".tmp{os.getpid()}"
        s.write(tmp)
        os.replace(tmp, path)
    return path


def frame_case(name):
    """Scene file, camera and render settings of one Part A scene."""
    if name.startswith("seed"):
        seed = int(name[4:])
        k = case_settings(seed)
        return dict(path=opaque_fuzz_scene(seed), cam=k["cam"], w=k["w"], h=k["h"], spp=k["spp"], first=k["first"], max=k["max"],
                    depth=k["depth"], bg=k["bg"], tonemap=TM[k["tonemap"]], tile=k["tile"])
    if name == "mclaren_200k":
        kw = dict(n_tris=200_000, env_res=256)
        return dict(path=H.scene_file("mclaren", **kw), cam=H.scene_camera("mclaren", **kw), w=320, h=180, spp=2, first=1, max=1,
                    depth=12, bg=(0.0, 0.0, 0.0), tonemap=Y.TONEMAP_AGX, tile=64)
    g = PC.load(os.path.join(H.GOLDEN, name))
    assert "integrator" not in g.files  # MIS: naiveStage has no walk parameter and always walks the BVH2
    scene, kw = PC.scene_from_golden(g)
    w, h, spp, first, mx, depth = (int(v) for v in g["settings"])
    return dict(path=H.scene_file(scene, **kw), cam=H.scene_camera(scene, **kw), w=w, h=h, spp=spp, first=first, max=mx, depth=depth,
                bg=(0.0, 0.0, 0.0), tonemap=PC.TONEMAPS[str(g["tonemap"])], tile=64)


def waves(c):
    """The wave sizes yr_render uses for these settings (tile-renderer.hpp's schedule, host/api.cpp)."""
    out, left = [], c["spp"]
    ws = min(c["first"] or left, left)
    mx = c["max"] or left
    while ws > 0:
        out.append(ws)
        left -= ws
        ws = min(min(ws * 2, mx) if (len(out) > 1 or ws > 1) else 1, left)
    return out


def camera(c):
    cam = c["cam"]
    return Y.make_camera(c["w"], c["h"], cam["focal"], cam["fnum"], cam["pos"], cam["target"], (0, 0, 0), cam["exposure"],
                         cam.get("sides", 0))


def small_capacity(c):
    """A wavefront capacity that cuts every sample of the frame into about six pixel blocks (two lanes)."""
    return c["w"] * c["h"] // 3


def counts(st):
    return int(st.raysReference), int(st.raysExtend), int(st.raysShadow)


def new_context(c, sc, traversal, shard=(0, 1), **opts):
    ctx = Y.Context(max_depth=c["depth"], traversal=traversal, **opts)
    ctx.upload_scene(sc)
    ctx.set_camera(camera(c))
    ctx.begin_frame(c["w"], c["h"], c["spp"], c["tile"], c["bg"], c["tonemap"], shard_index=shard[0], shard_count=shard[1])
    return ctx


def render(c, traversal=Y.TRAVERSAL_AUTO, async_waves=False, shard=(0, 1), **opts):
    """The frame through yc_render_wave (or yc_render_wave_async + yc_wave_sync): (hdr, ldr, ray counts)."""
    sc = Y.Scene(c["path"])
    ctx = new_context(c, sc, traversal, shard, **opts)
    taken = 0
    for wv in waves(c):
        (ctx.render_wave_async if async_waves else ctx.render_wave)(taken, wv, taken)
        taken += wv
    if async_waves:
        ctx.wave_sync()
    hdr, ldr, st = ctx.resolve()
    ctx.close()
    return hdr, ldr, counts(st)


def render_tile_shards(c, n=3):
    """n tile shards of the frame, summed (each shard's frames are zero outside its tiles)."""
    parts = [render(c, shard=(k, n)) for k in range(n)]
    return (functools.reduce(operator.add, (p[0] for p in parts)), functools.reduce(operator.add, (p[1] for p in parts)),
            tuple(map(sum, zip(*(p[2] for p in parts)))))


def render_bucket_shards(c, n=3):
    """n contexts each take the samples of every n-th estimator bucket (yc_accumulate_wave); their accumulation
    buffers are added as int32, as the multi-GPU all-reduce does, and finalized on every context."""
    sc = Y.Scene(c["path"])
    ctxs = [new_context(c, sc, Y.TRAVERSAL_AUTO) for _ in range(n)]
    taken = 0
    for wv in waves(c):
        total = None
        for g, ctx in enumerate(ctxs):
            ctx.accumulate_wave(taken, wv, bucket_shard=g, bucket_shard_count=n)
            ptr, nbytes, _, _ = ctx.bucket_device_ptrs()
            acc = np.empty(nbytes // 4, np.int32)
            ctx.d2h(acc, ptr)
            total = acc if total is None else total + acc
        for ctx in ctxs:
            ctx.h2d(ctx.bucket_device_ptrs()[0], total)
            ctx.finalize_wave(wv, taken)
        taken += wv
    out = [ctx.resolve() for ctx in ctxs]
    for ctx in ctxs:
        ctx.close()
    hdr, ldr, _ = out[0]
    for k, (h, l, _) in enumerate(out[1:], 1):
        assert H.bits_equal(h, hdr).all() and H.bits_equal(l, ldr).all(), f"bucket shard {k} finalized another frame than shard 0"
    return hdr, ldr, tuple(map(sum, zip(*(counts(st) for _, _, st in out))))


def render_renderer(c, **kw):
    """The frame through yr_render_sync (Renderer): one context, or several with `devices=` and `sharding=`."""
    sc = Y.Scene(c["path"])
    r = Y.Renderer(c["w"], c["h"], camera(c), sc, samples=c["spp"], first_wave_samples=c["first"], max_wave_samples=c["max"],
                   tile_size=c["tile"], max_depth=c["depth"], background=c["bg"], tonemap=c["tonemap"], traversal=Y.TRAVERSAL_AUTO, **kw)
    r.render_sync()
    hdr, ldr, st = r.read()
    r.close()
    return hdr, ldr, counts(st)


def assert_same_frame(tag, got, want):
    (hdr, ldr, rays), (hdr0, ldr0, rays0) = got, want
    bad = ~H.bits_equal(hdr, hdr0).all(-1)
    assert not bad.any(), f"{tag}: HDR differs in {bad.sum()} pixels, e.g. (y, x) {np.argwhere(bad)[:4].tolist()}"
    bad = ~H.bits_equal(ldr, ldr0).all(-1)
    assert not bad.any(), f"{tag}: LDR differs in {bad.sum()} pixels"
    assert rays == rays0, f"{tag}: rays (reference, extend, shadow) {rays} vs {rays0}"


def assert_wide(c):
    sc = Y.Scene(c["path"])
    ctx = Y.Context(max_depth=1, traversal=Y.TRAVERSAL_AUTO)
    ctx.upload_scene(sc)
    assert wide_active(ctx), f"{c['path']}: TRAVERSAL_AUTO does not run the wide walk on this scene"
    ctx.close()


def with_cpu_build(fn, *a, **kw):
    """fn run with the CPU build of the product sources bound; the library bound before is bound again afterwards."""
    lib = Y.lib()
    Y.use_library(H.hostsim())
    try:
        return fn(*a, **kw)
    finally:
        Y.use_library(lib)


@pytest.mark.parametrize("name", CASES)
def test_default_walk_frame_cpu_build(name, hostsim_lib):
    """The scene runs the wide walk under AUTO; AUTO equals an explicit TRAVERSAL_WIDE, the Renderer's frame equals
    yc_render_wave over the same waves (so one reference serves every configuration on the GPU), and the frame does
    not depend on the wavefront capacity."""
    c = frame_case(name)
    assert_wide(c)
    ref = render(c)
    assert np.nanmax(ref[0][..., :3]) > 0  # (frames of the "punchy" AgX look hold NaNs, as the reference's do)
    assert_same_frame(f"{name}, TRAVERSAL_WIDE", render(c, Y.TRAVERSAL_WIDE), ref)
    assert_same_frame(f"{name}, Renderer", render_renderer(c), ref)
    assert_same_frame(f"{name}, max_paths {small_capacity(c)}", render(c, max_paths=small_capacity(c)), ref)


# one capacity or tail variant per scene, in turn, besides the default context
VARIANTS = [dict(tail_threshold=-1), dict(max_paths=None), dict(sh_stack_entries=2), dict(tail_threshold=65536)]


@pytest.mark.gpu
@pytest.mark.parametrize("name", CASES)
def test_cuda_frames_equal_the_cpu_build_gpu(name, cuda_lib):
    """The CUDA library's frame equals the CPU build's under AUTO (default context and one variant) and under
    TRAVERSAL_REFERENCE_ORDER."""
    c = frame_case(name)
    ref, ref_order = with_cpu_build(lambda: (render(c), render(c, Y.TRAVERSAL_REFERENCE_ORDER)))
    assert_wide(c)
    assert_same_frame(f"{name}, default context", render(c), ref)
    opts = dict(VARIANTS[CASES.index(name) % len(VARIANTS)])
    if "max_paths" in opts:
        opts["max_paths"] = small_capacity(c)
    assert_same_frame(f"{name}, {opts}", render(c, **opts), ref)
    assert_same_frame(f"{name}, reference order", render(c, Y.TRAVERSAL_REFERENCE_ORDER), ref_order)


@pytest.mark.gpu
@pytest.mark.parametrize("name", FULL)
def test_cuda_frames_equal_the_cpu_build_in_every_configuration_gpu(name, cuda_lib):
    c = frame_case(name)
    ref = with_cpu_build(render, c)
    cap = small_capacity(c)
    configs = {
        "default context": lambda: render(c),
        "tail_threshold -1 (every bounce in the persistent kernels)": lambda: render(c, tail_threshold=-1),
        "tail_threshold 65536 (tail kernel from the second bounce)": lambda: render(c, tail_threshold=65536),
        f"max_paths {cap}": lambda: render(c, max_paths=cap),
        "2 shared stack entries (spill path)": lambda: render(c, sh_stack_entries=2),
        "waves left in flight": lambda: render(c, async_waves=True),
        f"waves left in flight, max_paths {cap}, tail_threshold 65536": lambda: render(c, async_waves=True, max_paths=cap,
                                                                                        tail_threshold=65536),
        "3 tile shards summed": lambda: render_tile_shards(c, 3),
        "3 bucket shards combined": lambda: render_bucket_shards(c, 3),
    }
    for n in (2, 3):
        for sharding, what in ((Y.SHARD_TILES, "tiles"), (Y.SHARD_BUCKETS, "buckets")):
            configs[f"Renderer over {n} contexts, {what}"] = lambda n=n, s=sharding: render_renderer(c, devices=devices(n), sharding=s)
    for tag, fn in configs.items():
        assert_same_frame(f"{name}, {tag}", fn(), ref)


# ------------------------------------------------------------------------------------------
# Part B: NEE transparency through stacks of thin panes, against float64
# ------------------------------------------------------------------------------------------
# layouts: all panes, the occluder and the wall in one mesh; one mesh per pane; one pane mesh instanced through K node
# transforms (translations); the same through a nested chain of K nodes.  The chain's steps turn the pane a quarter turn
# about the stack axis and scale it by 2 and 1/2 in turn: exact in float32, so the object-space direction the library
# forms is the float64 one and the bound below needs no transform term (test_wide_bvh_robustness covers general
# transforms for hit finding).
PANE_CASES = [dict(layout="one_mesh", k=k) for k in (1, 2, 3, 12, 64)] + \
             [dict(layout="per_pane", k=k) for k in (3, 12, 64)] + \
             [dict(layout="instanced", k=k) for k in (2, 12, 64)] + \
             [dict(layout="chain", k=k) for k in (3, 12)] + \
             [dict(layout=lay, k=12, offset=1e4) for lay in ("one_mesh", "instanced", "chain")] + \
             [dict(layout=lay, k=12, grazing=True) for lay in ("one_mesh", "per_pane")]


def pane_id(p):
    return f"{p['layout']}-k{p['k']}" + ("-far" if p.get("offset") else "") + ("-grazing" if p.get("grazing") else "")


SPACING = 0.25  # between neighbouring panes
ROT_Z90 = np.array([[0, -1, 0, 0], [1, 0, 0, 0], [0, 0, 1, 0], [0, 0, 0, 1]], np.float32)


def pane_scene(layout, k, offset=0.0, grazing=False, seed=0):
    """K thin transmissive panes (z = 0, SPACING, ...) with distinct base colours, half of them with an opaque base
    texture read at uv 0, an opaque wall behind the stack and an opaque occluder over part of the stack's middle gap.
    Returns the scene, the triangles for the float64 reference — (object-space vertices, object-space normal, world
    matrix, per-channel factor or None for opaque) — and the extent rays are aimed at."""
    rng = np.random.default_rng(100 + seed)
    half = 40.0 if grazing else 8.0
    s = scenes.Scene()
    texel = np.array([200, 120, 235], np.uint8)
    s.textures = [scenes.Texture(np.broadcast_to(np.append(texel, np.uint8(255)), (2, 2, 4)).copy(), scenes.SRGB)]
    tex_value = (texel.astype(np.float64) / 255.0) ** 2  # sRGB texels are stored squared (texture.cuh)
    n_mats = 1 if layout in ("instanced", "chain") else k  # instances share their mesh's material
    bases = rng.uniform(0.3, 0.95, (n_mats, 3)).astype(np.float32)
    factors = []
    for m in range(n_mats):
        textured = m % 2 == 1 or n_mats == 1
        s.materials.append(scenes.Material(base=tuple(bases[m]), base_tex=0 if textured else -1, transmission=float(rng.uniform(0.3, 1.0)),
                                           roughness=0.0, ior=1.5, thin=1))
        factors.append(bases[m].astype(np.float64) * (tex_value if textured else 1.0))
    opaque = len(s.materials)
    s.materials.append(scenes.Material(base=(0.5, 0.5, 0.5), roughness=1.0))
    off = np.array([offset, 0.5 * offset, 0.0])

    def pane(b, z, mat, h=half, shift=(0.0, 0.0, 0.0)):
        x0, y0 = shift[0] - h, shift[1] - h
        x1, y1 = shift[0] + h, shift[1] + h
        b.quad((x0, y0, z + shift[2]), (x1, y0, z + shift[2]), (x1, y1, z + shift[2]), (x0, y1, z + shift[2]), mat, uv_scale=0.0)

    # world z of the panes
    if layout == "chain":
        # step j: SPACING or 2 SPACING further along the parent's z, a quarter turn about z, a scale of 2 or 1/2
        local = [(scenes.translation(0.125, -0.0625, SPACING * (1 + j % 2)) if j else np.eye(4, dtype=np.float32)) @ ROT_Z90 @
                 scenes.scaling(2.0 if j % 2 == 0 else 0.5) for j in range(k)]
        chain = list(itertools.accumulate((x.astype(np.float64) for x in local), np.matmul))
        zs = [m[2, 3] for m in chain]
    else:
        zs = [j * SPACING for j in range(k)]
    z_wall = zs[-1] + 1.0 + 0.5 * (zs[-1] - zs[0])  # room behind the stack for tMax to end in
    z_occ = 0.5 * (zs[k // 2 - 1] + zs[k // 2]) if k >= 2 else None

    statics = scenes.MeshBuilder()  # the wall (and the occluder), in world coordinates
    pane(statics, z_wall, opaque, h=4 * half, shift=off)
    if z_occ is not None:
        statics.quad(off + (-0.4 * half, 0.0, z_occ), off + (0.4 * half, 0.0, z_occ), off + (0.4 * half, 0.6 * half, z_occ),
                     off + (-0.4 * half, 0.6 * half, z_occ), opaque)
    nodes = [scenes.Node(-1, -1)]
    world = {}  # node index → world matrix (float64)
    if layout in ("one_mesh", "per_pane"):
        builders = [scenes.MeshBuilder() for _ in range(1 if layout == "one_mesh" else k)]
        for j in range(k):
            pane(builders[0 if layout == "one_mesh" else j], zs[j], j, shift=off)
        if layout == "one_mesh":  # panes, occluder and wall in one BVH
            b = builders[0]
            st = statics.build()
            for f in st.faces:
                b.tri(*(st.positions[f[:3]].astype(np.float64)), int(f[3]))
            s.meshes = [b.build()]
        else:
            s.meshes = [b.build() for b in builders] + [statics.build()]
        for mi in range(len(s.meshes)):
            nodes.append(scenes.Node(0, mi))
            world[len(nodes) - 1] = np.eye(4)
    else:
        b = scenes.MeshBuilder()
        pane(b, 0.0, 0)
        s.meshes = [b.build(), statics.build()]
        nodes.append(scenes.Node(0, 1))
        world[1] = np.eye(4)
        parent, base = 0, np.eye(4)
        if offset:
            nodes.append(scenes.Node(0, -1, scenes.translation(*off)))
            parent, base = len(nodes) - 1, scenes.translation(*off).astype(np.float64)
        for j in range(k):
            if layout == "instanced":
                xf = scenes.translation(0.0, 0.0, zs[j])
                nodes.append(scenes.Node(parent, 0, xf))
                world[len(nodes) - 1] = base @ xf.astype(np.float64)
            else:
                nodes.append(scenes.Node(parent, 0, local[j]))
                parent = len(nodes) - 1
                world[parent] = base @ chain[j]
    s.nodes = nodes
    s.camera = dict(pos=(0.0, 0.0, -5.0), target=(0.0, 0.0, 0.0), focal=35.0, fnum=0.0, exposure=0.0, w=8, h=8, spp=1)
    tris = []
    for ni, m in world.items():
        mesh = s.meshes[s.nodes[ni].mesh]
        for f in mesh.faces:
            mat = int(f[3])
            tris.append((mesh.positions[f[:3]].astype(np.float64), mesh.normals[f[0]].astype(np.float64), m,
                         None if mat == opaque else factors[mat]))
    return s, tris, dict(z0=zs[0], z1=zs[-1], z_wall=z_wall, half=half, off=off)


def pane_rays(ext, n, grazing, seed=0):
    """Rays through the middle of the stack inside the panes: most run forward from in front of or inside the stack,
    some run back through it from behind; tMax ends anywhere from before the first pane to past the wall."""
    rng = np.random.default_rng(200 + seed)
    cz = rng.uniform(0.05, 0.3, n) if grazing else rng.uniform(0.25, 1.0, n)  # |d.z| = |n·d| at the panes
    phi = rng.uniform(0.0, 2 * np.pi, n)
    back = rng.uniform(size=n) < 0.15
    d = np.stack([np.sqrt(1 - cz * cz) * np.cos(phi), np.sqrt(1 - cz * cz) * np.sin(phi), np.where(back, -cz, cz)], 1)
    zm = 0.5 * (ext["z0"] + ext["z1"])
    front = rng.uniform(size=n) < 0.5  # forward rays from in front of the stack, or from inside its first half
    oz = np.where(back, rng.uniform(zm, ext["z_wall"] - 0.1, n),
                  np.where(front, rng.uniform(ext["z0"] - 1.0, ext["z0"], n), rng.uniform(ext["z0"], zm, n)))
    target = np.stack([rng.uniform(-0.7, 0.7, n) * ext["half"], rng.uniform(-0.7, 0.7, n) * ext["half"], np.full(n, zm)], 1)
    o = target - d * ((zm - oz) / d[:, 2])[:, None]
    t_end = np.where(back, (oz - ext["z0"] + 1.0) / cz, (ext["z_wall"] - oz) / cz)
    rays = np.zeros((n, 8), np.float32)
    rays[:, :3] = o + ext["off"]
    rays[:, 3] = KTMIN
    rays[:, 4:7] = d
    rays[:, 7] = t_end * rng.uniform(0.05, 1.15, n)
    return rays


def pane_reference(tris, rays):
    """float64: (rays kept, occluded, attenuation, panes crossed).  A ray is occluded when an opaque triangle has t in
    (kTMin, tMax); otherwise its attenuation is the product of |n·d|·base over the panes with t in that range, n and d
    in the pane's object space (testTriangle: the interpolated normal against the untransformed-length object-space
    direction).  Rays within a relative margin of tMax or kTMin, or of a triangle's edges (the quads' diagonals
    included), or nearly parallel to a triangle they reach, are left out."""
    o, d, tmax = rays[:, :3].astype(np.float64), rays[:, 4:7].astype(np.float64), rays[:, 7].astype(np.float64)
    n = len(rays)
    keep, occ = np.ones(n, bool), np.zeros(n, bool)
    att, crossed = np.ones((n, 3)), np.zeros(n, int)
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        for (p, nrm, m, factor) in tris:
            inv = np.linalg.inv(m)
            oo, dd = o @ inv[:3, :3].T + inv[:3, 3], d @ inv[:3, :3].T
            e1, e2 = p[1] - p[0], p[2] - p[0]
            pv = np.cross(dd, e2)
            det = pv @ e1
            s = oo - p[0]
            u = np.einsum("ij,ij->i", s, pv) / det
            qv = np.cross(s, e1)
            v = np.einsum("ij,ij->i", dd, qv) / det
            t = (qv @ e2) / det
            bmin = np.minimum(np.minimum(u, v), 1.0 - u - v)
            scale = np.abs(oo).max(1) + np.abs(p).max()
            mb = 1e-4 + 1e-6 * scale / min(np.linalg.norm(e1), np.linalg.norm(e2))
            mt = 1e-4 * np.abs(t) + 1e-6 * scale / np.linalg.norm(dd, axis=1)
            cos = np.abs(det) / (np.linalg.norm(np.cross(e1, e2)) * np.linalg.norm(dd, axis=1))
            reach = (bmin > -mb) & (t > KTMIN - mt) & (t < tmax + mt)
            keep &= ~(reach & ((bmin < mb) | (np.abs(t - tmax) <= mt) | (np.abs(t - KTMIN) <= mt) | (cos < 0.02)))
            hit = (bmin >= mb) & (t > KTMIN) & (t < tmax)
            if factor is None:
                occ |= hit
            else:
                att[hit] *= np.abs(dd[hit] @ nrm)[:, None] * factor
                crossed += hit
    return keep, occ, att, crossed


def trace_panes(path, rays):
    """Any-hit records of both walks (TRACE_WIDE, TRACE_REFERENCE_ORDER) on an AUTO context."""
    sc = Y.Scene(path)
    ctx = Y.Context(max_depth=1, traversal=Y.TRAVERSAL_AUTO)
    ctx.upload_scene(sc)
    assert wide_active(ctx)
    out = {walk: ctx.trace(rays, Y.TRACE_ANY | walk)[0] for walk in (Y.TRACE_WIDE, Y.TRACE_REFERENCE_ORDER)}
    ctx.close()
    return out


def check_panes(p, tmp_path):
    """Both walks of the active library against the float64 reference; returns the scene file, rays and records."""
    s, tris, ext = pane_scene(p["layout"], p["k"], p.get("offset", 0.0), p.get("grazing", False))
    path = str(tmp_path / f"{pane_id(p)}.ysc")
    s.write(path)
    rays = pane_rays(ext, 4000, p.get("grazing", False))
    keep, occ, att, crossed = pane_reference(tris, rays)
    k = p["k"]
    free = keep & ~occ
    # enough of every kind: kept rays, occluded ones, and unoccluded ones through panes (through all K for small K)
    assert keep.mean() > 0.5 and (keep & occ).sum() > 50 and (free & (crossed > 0)).sum() > 300, (keep.sum(), (keep & occ).sum())
    assert (free & (crossed == k)).sum() >= 10
    measured = free & (att.min(1) > 1e-30)  # float32 attenuation still normal with room to spare
    bound = (3 * k + 8) * U
    out = trace_panes(path, rays)
    for walk, hits in out.items():
        tag = f"{pane_id(p)}, {'wide' if walk == Y.TRACE_WIDE else 'reference-order'} walk"
        did = hits["didHit"] == 1
        wrong = keep & (did != occ)
        assert not wrong.any(), (f"{tag}: occlusion differs from float64 on {wrong.sum()} of {keep.sum()} rays, e.g. {np.nonzero(wrong)[0][:5]}"
                                 f" (float64 occluded {occ[wrong][:5]}, panes crossed {crossed[wrong][:5]})")
        rel = np.abs(hits["attenuation"][measured].astype(np.float64) - att[measured]) / att[measured]
        worst = rel.max(initial=0.0)
        print(f"{tag}: {keep.sum()} rays kept, {(keep & occ).sum()} occluded, {measured.sum()} attenuations checked, "
              f"largest relative error {worst / U:.1f} u (bound {3 * k + 8} u)")
        if worst > bound:
            i = np.nonzero(measured)[0][rel.max(1).argmax()]
            raise AssertionError(f"{tag}: attenuation off by {worst:.3g} relative (bound {bound:.3g}) on ray {i}: "
                                 f"{hits['attenuation'][i]} vs {att[i]}, {crossed[i]} panes crossed")
    return path, rays, out


@pytest.mark.parametrize("p", PANE_CASES, ids=pane_id)
def test_nee_transparency_matches_float64_cpu_build(p, tmp_path, hostsim_lib):
    check_panes(p, tmp_path)


@pytest.mark.gpu
@pytest.mark.parametrize("p", PANE_CASES, ids=pane_id)
def test_nee_transparency_matches_float64_and_the_cpu_build_gpu(p, tmp_path, cuda_lib):
    path, rays, got = check_panes(p, tmp_path)
    want = with_cpu_build(trace_panes, path, rays)
    for walk in got:
        differ = (got[walk].view(np.uint8).reshape(len(rays), -1) != want[walk].view(np.uint8).reshape(len(rays), -1)).any(1)
        assert not differ.any(), f"{pane_id(p)}, walk {walk:#x}: CUDA any-hit records differ from the CPU build's on {differ.sum()} rays"
