"""The 4-wide collapsed BVH (yart_b200/csrc/wide_bvh.cuh, YC_TRAVERSAL_WIDE / the AUTO default for scenes without
alpha-tested materials) against the reference's recorded outputs, with the north-star bars: identical rays → hit
triangle ids exact except documented ties (same t to the last bit on another triangle), t within 1e-5 relative
(in fact bit-exact: the triangle arithmetic is the reference's), frames relMSE < 1e-3 on HDR and after AgX.

CPU part: the product sources compiled for the CPU (tests/hostsim; sequential walk testBVHWide).  The `-m gpu` part
runs the persistent-warp kernels (tracePersistent over WideWalk, trace_kernels.cuh) through the same checks."""
import os

import numpy as np
import pytest

import harness as H
import parity_common as PC
import yart_b200 as Y

WIDE_TRACE_SCENES = ("cornell", "mclaren", "soup", "two_quads")  # trace goldens of scenes without alpha-tested materials
WIDE_RENDER = ("render_cornell.npz", "render_cornell_waves.npz", "render_mclaren_small.npz", "render_soup_d1.npz",
               "render_two_quads.npz")


def check_trace_wide(path):
    g = PC.load(path)
    name, kw = PC.scene_from_golden(g)
    sc = Y.Scene(H.scene_file(name, **kw))
    ctx = Y.Context(traversal=Y.TRAVERSAL_WIDE)
    ctx.upload_scene(sc)
    rays = g["rays"]
    ref = g["closest"]
    hits, _ = ctx.trace(rays, Y.TRACE_CLOSEST)
    assert np.array_equal(hits["didHit"], ref["didHit"]), f"{name}: didHit differs"
    m = ref["didHit"] == 1
    rel = np.abs(hits["t"][m] - ref["t"][m]) / np.abs(ref["t"][m])
    assert rel.max(initial=0.0) <= 1e-5
    other = m & (hits["prim"] != ref["prim"])
    # documented ties: another triangle with the SAME t (bitwise) — e.g. a ray through the diagonal of a quad
    assert np.array_equal(hits["t"][other].view(np.uint32), ref["t"][other].view(np.uint32)), f"{name}: id differs without a tie"
    assert other.sum() <= max(2, len(rays) // 500), f"{name}: {other.sum()} ties"
    same = m & ~other
    for f in ("t", "material", "lightIdx", "backSide", "p", "n", "tg", "uv"):
        assert np.array_equal(hits[f][same].view(np.uint32), ref[f][same].view(np.uint32)), f"{name}: Hit::{f} differs"
    ref_any = g["anyhit"]
    anyh, _ = ctx.trace(rays, Y.TRACE_ANY)
    assert np.array_equal(anyh["didHit"], ref_any["didHit"]), f"{name}: any-hit result differs"
    free = ref_any["didHit"] == 0  # Hit::attenuation only matters for unoccluded rays; product order may differ
    assert np.allclose(anyh["attenuation"][free], ref_any["attenuation"][free], rtol=1e-5, atol=0)
    # the forced-mode bits agree with the context modes
    h_ref, _ = ctx.trace(rays, Y.TRACE_CLOSEST | Y.TRACE_REFERENCE_ORDER)
    assert np.array_equal(h_ref["prim"], ref["prim"]) and np.array_equal(h_ref["t"].view(np.uint32), ref["t"].view(np.uint32))
    _, st_w = ctx.trace(rays, Y.TRACE_CLOSEST | Y.TRACE_COUNT | Y.TRACE_WIDE)
    _, st_r = ctx.trace(rays, Y.TRACE_CLOSEST | Y.TRACE_COUNT)
    assert st_w.boxTests > 0 and st_r.boxTests > 0 and st_w.triTests > 0
    ctx.close()
    return int(other.sum())


def check_render_wide(path):
    g, data, hdr, ldr, st = PC.render_golden(path, traversal=Y.TRAVERSAL_WIDE)
    tag = os.path.basename(path)
    rh, rl = H.rel_mse(hdr, g["hdr"]), H.rel_mse(ldr, g["ldr"])
    assert rh < 1e-3 and rl < 1e-3, f"{tag}: relMSE hdr {rh} ldr {rl}"
    assert abs(int(data["total_rays"]) - int(g["rays"])) <= 1e-3 * int(g["rays"])
    same = H.bits_equal(hdr, g["hdr"]).all(-1).mean()
    assert same > 0.995, f"{tag}: only {same:.5f} of the pixels are bit-identical to the reference"
    return same


@pytest.mark.parametrize("scene", WIDE_TRACE_SCENES)
def test_wide_trace_cpu_build(scene, hostsim_lib):
    check_trace_wide(os.path.join(H.GOLDEN, f"trace_{scene}.npz"))


@pytest.mark.parametrize("name", WIDE_RENDER)
def test_wide_render_cpu_build(name, hostsim_lib):
    check_render_wide(os.path.join(H.GOLDEN, name))


def _axis_rays():
    """Rays with zero direction components and origins on those planes: the reference's slab test is NaN there."""
    rays = []
    for y in np.linspace(-8, 8, 9):
        for z in (-1.0, 0.0, 1.0):
            rays.append([0.0, y, 40.0, 0.001, 0.0, 0.0, -1.0, np.inf])       # d.x = d.y = 0, o.x = 0
            rays.append([0.0, 0.0, 40.0, 0.001, 0.0, y / 40.0, -1.0, np.inf])  # d.x = 0, o.x = o.y = 0
            rays.append([z, y, 0.0, 0.001, 0.0, 1.0, 0.0, np.inf])           # along +y from inside the soup
    r = np.asarray(rays, np.float32)
    r[:, 4:7] /= np.linalg.norm(r[:, 4:7], axis=1, keepdims=True)
    return r


def _check_axis_rays():
    sc = Y.Scene(H.scene_file("soup", n_tris=20_000))
    ctx = Y.Context(max_depth=1, traversal=Y.TRAVERSAL_WIDE)
    ctx.upload_scene(sc)
    rays = _axis_rays()
    ref, st_r = ctx.trace(rays, Y.TRACE_CLOSEST | Y.TRACE_COUNT | Y.TRACE_REFERENCE_ORDER)
    wide, st_w = ctx.trace(rays, Y.TRACE_CLOSEST | Y.TRACE_COUNT | Y.TRACE_WIDE)
    assert np.array_equal(wide["didHit"], ref["didHit"]) and np.array_equal(wide["prim"], ref["prim"])
    assert np.array_equal(wide["t"].view(np.uint32), ref["t"].view(np.uint32))
    # the clamped reciprocal direction removes the walk over every box overlapping the ray's plane
    assert st_w.boxTests * 4 < st_r.boxTests, (st_w.boxTests, st_r.boxTests)
    ctx.close()


def test_wide_axis_aligned_rays_same_hits_far_fewer_boxes_cpu_build(hostsim_lib):
    _check_axis_rays()


def test_wide_is_refused_for_alpha_scenes_and_auto_falls_back(hostsim_lib):
    sc = Y.Scene(H.scene_file("material_zoo"))
    ctx = Y.Context(traversal=Y.TRAVERSAL_WIDE)
    with pytest.raises(Y.YartError, match="UNSUPPORTED"):
        ctx.upload_scene(sc)
    ctx.close()
    # AUTO on an alpha scene is the reference-order walk: bit-identical to the golden
    g, data, hdr, ldr, st = PC.render_golden(os.path.join(H.GOLDEN, "render_zoo.npz"), traversal=Y.TRAVERSAL_AUTO)
    assert H.bits_equal(hdr, g["hdr"]).all() and data["total_rays"] == int(g["rays"])
    ctx = Y.Context(traversal=Y.TRAVERSAL_AUTO)
    ctx.upload_scene(sc)
    with pytest.raises(Y.YartError, match="STATE"):
        ctx.trace(np.zeros((1, 8), np.float32), Y.TRACE_CLOSEST | Y.TRACE_WIDE)
    ctx.close()


def test_wide_deep_path_render_with_tail_kernel_and_chunking_cpu_build(hostsim_lib):
    """Full MIS+NEE paths through the wide walk, small wavefront capacity (many chunks): equal to the single-chunk render."""
    path = os.path.join(H.GOLDEN, "render_mclaren_small.npz")
    g = PC.load(path)
    name, kw = PC.scene_from_golden(g)
    w, h, spp, first, mx, depth = (int(v) for v in g["settings"])
    cam = H.scene_camera(name, **kw)
    sc = Y.Scene(H.scene_file(name, **kw))
    c = Y.make_camera(w, h, cam["focal"], cam["fnum"], cam["pos"], cam["target"], (0, 0, 0), cam["exposure"])
    out = []
    for cap in (0, 2048):
        ctx = Y.Context(max_depth=depth, max_paths=cap, traversal=Y.TRAVERSAL_WIDE)
        ctx.upload_scene(sc)
        ctx.set_camera(c)
        ctx.begin_frame(w, h, spp, 64, (0, 0, 0), Y.TONEMAP_AGX)
        ctx.render_wave(0, spp, 0)
        hdr, _, st = ctx.resolve()
        out.append((hdr, st.raysReference))
        ctx.close()
    assert H.bits_equal(out[0][0], out[1][0]).all() and out[0][1] == out[1][1]


# ------------------------------------------------------------------------------------------
# the same on the GPU (persistent-warp kernels)
# ------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("scene", WIDE_TRACE_SCENES)
def test_wide_trace_gpu(scene, cuda_lib):
    check_trace_wide(os.path.join(H.GOLDEN, f"trace_{scene}.npz"))


@pytest.mark.gpu
@pytest.mark.parametrize("name", WIDE_RENDER)
def test_wide_render_gpu(name, cuda_lib):
    check_render_wide(os.path.join(H.GOLDEN, name))


@pytest.mark.gpu
def test_wide_axis_aligned_rays_gpu(cuda_lib):
    _check_axis_rays()


@pytest.mark.gpu
def test_wide_gpu_kernels_equal_the_cpu_build_of_the_same_sources(cuda_lib):
    """The persistent-warp wide kernels and the sequential walk make the same decisions (nearest child by key,
    slot-order pushes): hit records of 200 K primary rays of the 100 K soup are identical, ties included."""
    sc_path = H.scene_file("soup", n_tris=100_000)
    cam = H.scene_camera("soup")
    W, Hh = 640, 360
    recs = []
    for lib in (cuda_lib, H.hostsim()):
        Y.use_library(lib)
        sc = Y.Scene(sc_path)
        ctx = Y.Context(max_depth=1, traversal=Y.TRAVERSAL_WIDE)
        ctx.upload_scene(sc)
        ctx.set_camera(Y.make_camera(W, Hh, cam["focal"], cam["fnum"], cam["pos"], cam["target"]))
        ctx.begin_frame(W, Hh, 1, 64, (0, 0, 0), Y.TONEMAP_NONE)
        rays_dev = ctx.device_alloc(W * Hh * 32)
        ctx.generate_primary_rays(0, 1, rays_dev)
        rays = np.empty((W * Hh, 8), np.float32)
        ctx.d2h(rays, rays_dev)
        ctx.device_free(rays_dev)
        hits, _ = ctx.trace(rays, Y.TRACE_CLOSEST)
        anyh, _ = ctx.trace(np.concatenate([rays[:, :7], np.full((len(rays), 1), 30.0, np.float32)], 1), Y.TRACE_ANY)
        recs.append((rays.tobytes(), hits.tobytes(), anyh["didHit"].tobytes()))
        ctx.close()
    Y.use_library(cuda_lib)
    assert recs[0][0] == recs[1][0] and recs[0][1] == recs[1][1] and recs[0][2] == recs[1][2]


def test_wide_collapse_shared_out_over_threads_cpu_build(hostsim_lib):
    """A mesh big enough (>= 50 000 inner nodes) for the collapse to hand subtrees to worker threads and stitch the
    pieces: the wide walk finds what the reference-order walk finds (ids bar ties at the bit-identical t, t to 1e-5)."""
    sc = Y.Scene(H.scene_file("soup", n_tris=120_000))
    ctx = Y.Context(traversal=Y.TRAVERSAL_WIDE)
    ctx.upload_scene(sc)
    rng = np.random.default_rng(3)
    n = 20000
    o = rng.uniform(-12, 12, (n, 3)).astype(np.float32)
    d = rng.normal(size=(n, 3)).astype(np.float32)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    rays = np.concatenate([o, np.full((n, 1), 1e-4, np.float32), d, np.full((n, 1), np.inf, np.float32)], axis=1).astype(np.float32)
    wide, _ = ctx.trace(rays, Y.TRACE_CLOSEST)
    ref, _ = ctx.trace(rays, Y.TRACE_CLOSEST | Y.TRACE_REFERENCE_ORDER)
    assert np.array_equal(wide["didHit"], ref["didHit"]) and ref["didHit"].sum() > n // 4
    m = ref["didHit"] == 1
    assert (np.abs(wide["t"][m] - ref["t"][m]) <= 1e-5 * np.abs(ref["t"][m])).all()
    other = m & (wide["prim"] != ref["prim"])
    assert np.array_equal(wide["t"][other].view(np.uint32), ref["t"][other].view(np.uint32)) and other.sum() <= 4
    any_w, _ = ctx.trace(rays, Y.TRACE_ANY)
    any_r, _ = ctx.trace(rays, Y.TRACE_ANY | Y.TRACE_REFERENCE_ORDER)
    assert np.array_equal(any_w["didHit"], any_r["didHit"])
    ctx.close()
