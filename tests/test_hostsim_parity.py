"""CPU parity suite: the product sources compiled for the host (tests/hostsim, kernels as loops)
against the reference's recorded outputs.  Both sides use glibc's libm and no FMA contraction, so
EVERYTHING must be bit-exact here — any differing bit is a logic difference from the reference."""
import os

import numpy as np
import pytest

import harness as H
import parity_common as PC
import yart_b200 as Y

pytestmark = pytest.mark.usefixtures("hostsim_lib")


@pytest.mark.parametrize("path", PC.golden_files("kat"), ids=os.path.basename)
def test_kat_bit_exact(path):
    PC.check_kat(Y.Context, path, exact=True)


@pytest.mark.parametrize("path", PC.golden_files("bvh"), ids=os.path.basename)
def test_bvh_builder_reproduces_reference_tree(path):
    g = PC.load(path)
    name, kw = PC.scene_from_golden(g)
    sc = Y.Scene(H.scene_file(name, **kw))
    i = 0
    while f"nodes{i}" in g.files:
        nodes, idx = sc.bvh(i)
        assert nodes.tobytes() == g[f"nodes{i}"].tobytes(), f"{name} mesh {i}: nodes differ"
        assert np.array_equal(idx, g[f"idx{i}"]), f"{name} mesh {i}: index permutation differs"
        i += 1
    assert i == sc.flat.nMeshes


@pytest.mark.parametrize("path", PC.golden_files("variantkat"), ids=os.path.basename)
def test_variant_kat_bit_exact(path):
    """UniformLightSampler (light-sampler.cpp:11-31) against the reference's class."""
    PC.check_kat(Y.Context, path, exact=True)


@pytest.mark.parametrize("path", PC.golden_files("medianbvh"), ids=os.path.basename)
def test_median_split_builder_reproduces_reference_tree(path):
    """YS_BVH_MEDIAN_SPLIT against MedianSplitBVH (bvh.hpp:237-264) built by the oracle over the same meshes; a render
    through that tree must give the SAH tree's image (same triangles, same arithmetic per test; no ties in this scene)."""
    g = PC.load(path)
    name, kw = PC.scene_from_golden(g)
    sc = Y.Scene(H.scene_file(name, **kw), bvh_kind=Y.BVH_MEDIAN_SPLIT)
    i = 0
    while f"nodes{i}" in g.files:
        nodes, idx = sc.bvh(i)
        assert nodes.tobytes() == g[f"nodes{i}"].tobytes(), f"{name} mesh {i}: nodes differ"
        assert np.array_equal(idx, g[f"idx{i}"]), f"{name} mesh {i}: index permutation differs"
        i += 1
    assert i == sc.flat.nMeshes
    if name == "cornell":
        cam = H.scene_camera(name)
        c = Y.make_camera(32, 32, cam["focal"], cam["fnum"], cam["pos"], cam["target"])
        frames = []
        for scene in (sc, Y.Scene(H.scene_file(name, **kw))):
            ctx = Y.Context(max_depth=4)
            ctx.upload_scene(scene)
            ctx.set_camera(c)
            ctx.begin_frame(32, 32, 4, 64, (0, 0, 0), Y.TONEMAP_AGX)
            ctx.render_wave(0, 4, 0)
            frames.append(ctx.resolve()[0])
            ctx.close()
        assert H.bits_equal(frames[0], frames[1]).all()


@pytest.mark.parametrize("path", PC.golden_files("trace"), ids=os.path.basename)
def test_trace_bit_exact(path):
    PC.check_trace(Y.Context, path)


@pytest.mark.parametrize("path", PC.golden_files("render"), ids=os.path.basename)
def test_render_bit_exact(path):
    PC.check_render(path, exact=True)


@pytest.mark.parametrize("path", PC.golden_files("naive"), ids=os.path.basename)
def test_naive_integrator_render_bit_exact(path):
    """TileRenderer<SobolSampler<FastOwenScrambler>, NaiveIntegrator> (naive-integrator.cpp), progressive waves included."""
    PC.check_render(path, exact=True)


@pytest.mark.parametrize("path", PC.golden_files("scrambler"), ids=os.path.basename)
def test_other_scramblers_render_bit_exact(path):
    """TileRenderer<SobolSampler<OwenScrambler | BinaryPermuteScrambler>, MISIntegrator> (scrambler.hpp:35-85)."""
    PC.check_render(path, exact=True)


@pytest.mark.parametrize("path", PC.golden_files("sampler"), ids=os.path.basename)
def test_rng_samplers_render_bit_exact(path):
    """TileRenderer<NaiveSampler | StratifiedSampler, MISIntegrator> (sampler.cpp:5-50, xoshiro256++ + libstdc++'s
    uniform_real_distribution<float>), progressive waves included."""
    PC.check_render(path, exact=True)


def render_waves(g, **ctx_opts):
    """The golden's frame through one Context and yc_render_wave, in the golden's progressive waves: hdr, ldr, stats."""
    name, kw = PC.scene_from_golden(g)
    w, h, spp, first, mx, depth = (int(v) for v in g["settings"])
    cam = H.scene_camera(name, **kw)
    c = Y.make_camera(w, h, cam["focal"], cam["fnum"], cam["pos"], cam["target"], (0, 0, 0), cam["exposure"])
    ctx = Y.Context(max_depth=depth, **ctx_opts)
    ctx.upload_scene(Y.Scene(H.scene_file(name, **kw)))
    ctx.set_camera(c)
    ctx.begin_frame(w, h, spp, 64, (0, 0, 0), PC.TONEMAPS[str(g["tonemap"])])
    taken, wave, waves = 0, first, 0
    while wave > 0:
        ctx.render_wave(taken, wave, taken)
        taken += wave
        nxt = min(wave * 2, mx) if (waves > 0 or wave > 1) else 1
        wave = min(nxt, spp - taken)
        waves += 1
    hdr, ldr, st = ctx.resolve()
    ctx.close()
    return hdr, ldr, st


def test_small_wavefront_capacity_gives_same_image():
    """Chunking (pixel blocks x sample groups) must not change a single bit."""
    g = PC.load(os.path.join(H.GOLDEN, "render_cornell_waves.npz"))
    for cap in (700, 5000):  # < pixels (pixel blocks, K = 1) and ≈ 2.6 x pixels (K = 2)
        hdr, ldr, st = render_waves(g, max_paths=cap)
        assert H.bits_equal(hdr, g["hdr"]).all() and H.bits_equal(ldr, g["ldr"]).all()
        assert st.raysReference == int(g["rays"])


# (golden, traversal, whether the frame is the golden's): the tail runs as tailKernel<false, Bvh2Walk>,
# tailKernel<true, Bvh2Walk> (alpha-tested materials) and tailKernel<false, WideWalk>
TAIL_CASES = [("render_cornell_waves.npz", Y.TRAVERSAL_REFERENCE_ORDER, True), ("render_zoo.npz", Y.TRAVERSAL_REFERENCE_ORDER, True),
              ("render_mclaren_small.npz", Y.TRAVERSAL_WIDE, False)]


@pytest.mark.parametrize("name,traversal,golden", TAIL_CASES, ids=[c[0] for c in TAIL_CASES])
def test_tail_hand_over_gives_same_image(name, traversal, golden):
    """The per-path tail kernel that finishes a chunk once few paths survive must not change a single bit: tail never
    (-1), at the default threshold (0) and from the second bounce on (65536)."""
    g = PC.load(os.path.join(H.GOLDEN, name))
    out = {t: render_waves(g, traversal=traversal, tail_threshold=t) for t in (-1, 0, 65536)}
    hdr, ldr, st = out[-1]
    if golden:
        assert H.bits_equal(hdr, g["hdr"]).all() and H.bits_equal(ldr, g["ldr"]).all()
        assert st.raysReference == int(g["rays"])
    for t in (0, 65536):
        h, l, s = out[t]
        assert H.bits_equal(h, hdr).all() and H.bits_equal(l, ldr).all(), f"tail_threshold {t}: frame differs"
        assert (s.raysReference, s.raysExtend, s.raysShadow) == (st.raysReference, st.raysExtend, st.raysShadow)
    # the tail ran: it replaces the six launches of every later bounce by one
    assert out[65536][2].kernelLaunches < st.kernelLaunches


def test_tile_shards_sum_to_the_full_frame():
    """Interleaved tile sharding (SURVEY §8e): per-shard frames are disjoint, their sum is bit-identical."""
    path = os.path.join(H.GOLDEN, "render_zoo.npz")
    g = PC.load(path)
    parts = []
    rays = 0
    for k in range(3):
        _, data, hdr, ldr, _ = PC.render_golden(path, shard_index=k, shard_count=3, tile_size=16)
        parts.append((hdr, ldr))
        rays += data["total_rays"]
    hdr = parts[0][0] + parts[1][0] + parts[2][0]
    ldr = parts[0][1] + parts[1][1] + parts[2][1]
    # tile_size 16 changes the sampler's nBase4Digits, so compare with an unsharded tile-16 render
    _, data1, hdr1, ldr1, _ = PC.render_golden(path, tile_size=16)
    assert H.bits_equal(hdr, hdr1).all() and H.bits_equal(ldr, ldr1).all() and rays == data1["total_rays"]
    nz = [(p[0][..., 3] != 0) for p in parts]
    assert not (nz[0] & nz[1]).any() and not (nz[0] & nz[2]).any() and not (nz[1] & nz[2]).any()


def test_sub_rectangle_wave_matches_full_frame_pixels():
    path = os.path.join(H.GOLDEN, "render_two_quads.npz")
    g = PC.load(path)
    name, kw = PC.scene_from_golden(g)
    cam = H.scene_camera(name)
    sc = Y.Scene(H.scene_file(name))
    c = Y.make_camera(64, 64, cam["focal"], cam["fnum"], cam["pos"], cam["target"])
    ctx = Y.Context()
    ctx.upload_scene(sc)
    ctx.set_camera(c)
    ctx.begin_frame(64, 64, 16, 64, (0, 0, 0), Y.TONEMAP_AGX)
    ctx.render_wave(0, 16, 0, rect=(10, 20, 30, 17))
    hdr, _, _ = ctx.resolve()
    assert H.bits_equal(hdr[20:37, 10:40], g["hdr"][20:37, 10:40]).all()
    mask = np.ones((64, 64), bool)
    mask[20:37, 10:40] = False
    assert (hdr[mask] == 0).all()
