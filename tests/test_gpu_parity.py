"""GPU parity suite (`-m gpu`): libyart_b200.so (CUDA, sm_100a) through the C ABI against the
reference's recorded outputs (tests/golden) and size-independent properties at full frame sizes.

Bars (BASELINE.json north_star): identical rays → hit triangle IDs bit-exact, t within 1e-5 relative
(we get bit-exact: traversal is +,-,*,/ only, compiled -fmad=false); images at equal spp with the
reference's sampler streams → per-pixel relative MSE < 1e-3, HDR and after AgX."""
import os

import numpy as np
import pytest

import harness as H
import parity_common as PC
import yart_b200 as Y

pytestmark = [pytest.mark.gpu, pytest.mark.usefixtures("cuda_lib")]


def test_cuda_library_is_the_one_loaded():
    import yart_b200.capi as capi
    assert os.path.samefile(Y.lib()._name, capi.PRODUCT_LIB)
    ctx = Y.Context()  # raises without a device: no fallback
    ctx.close()


@pytest.mark.parametrize("path", PC.golden_files("kat"), ids=os.path.basename)
def test_kat(path):
    PC.check_kat(Y.Context, path, exact=False)


@pytest.mark.parametrize("path", PC.golden_files("trace"), ids=os.path.basename)
def test_trace_bit_exact(path):
    PC.check_trace(Y.Context, path)


@pytest.mark.parametrize("path", PC.golden_files("render"), ids=os.path.basename)
def test_render_rel_mse(path):
    PC.check_render(path, exact=False)


@pytest.mark.parametrize("path", PC.golden_files("naive"), ids=os.path.basename)
def test_naive_integrator_render(path):
    """YC_INTEGRATOR_NAIVE against TileRenderer<SobolSampler<FastOwenScrambler>, NaiveIntegrator> (relMSE < 1e-3, then bitwise)."""
    PC.check_render(path, exact=False)


@pytest.mark.parametrize("path", PC.golden_files("scrambler"), ids=os.path.basename)
def test_other_scramblers_render(path, cuda_samplers_lib):
    """YC_SCRAMBLER_OWEN / _BINARY_PERMUTE (libyart_b200_samplers.so) against TileRenderer<SobolSampler<R>, MISIntegrator> (relMSE < 1e-3, then bitwise)."""
    PC.check_render(path, exact=False)


@pytest.mark.parametrize("path", PC.golden_files("sampler"), ids=os.path.basename)
def test_rng_samplers_render(path, cuda_samplers_lib):
    """YC_SAMPLER_NAIVE / _STRATIFIED (libyart_b200_samplers.so) against TileRenderer<NaiveSampler | StratifiedSampler,
    MISIntegrator> (relMSE < 1e-3, then bitwise)."""
    PC.check_render(path, exact=False)


@pytest.mark.parametrize("path", PC.golden_files("variantkat"), ids=os.path.basename)
def test_variant_kat(path, cuda_samplers_lib):
    PC.check_kat(Y.Context, path, exact=True)


def test_uniform_light_sampler_renders_and_differs_only_in_noise(cuda_samplers_lib):
    """No frame of the reference exists for UniformLightSampler (MISIntegrator hard-codes PowerLightSampler); the
    render must run, stay finite, and agree with the power sampler's image on average (both are unbiased)."""
    name = "material_zoo"
    cam = H.scene_camera(name)
    sc = Y.Scene(H.scene_file(name))
    c = Y.make_camera(96, 54, cam["focal"], cam["fnum"], cam["pos"], cam["target"], (0, 0, 0), cam["exposure"])
    means = []
    for ls in (Y.LIGHT_SAMPLER_POWER, Y.LIGHT_SAMPLER_UNIFORM):
        ctx = Y.Context(max_depth=6, light_sampler=ls)
        ctx.upload_scene(sc)
        ctx.set_camera(c)
        ctx.begin_frame(96, 54, 64, 64, (0, 0, 0), Y.TONEMAP_AGX, estimator=Y.ESTIMATOR_MEAN)
        ctx.render_wave(0, 64, 0)
        hdr, _, _ = ctx.resolve()
        assert np.isfinite(hdr).all()
        means.append(hdr[..., :3].mean())
        ctx.close()
    assert abs(means[0] - means[1]) < 0.1 * means[0]


def test_default_library_refuses_rng_samplers_loudly():
    with pytest.raises(Y.YartError, match="UNSUPPORTED.*SAMPLERS_LIB"):
        Y.Context(sampler=Y.SAMPLER_NAIVE)
    with pytest.raises(Y.YartError, match="UNSUPPORTED"):
        Y.Context(scrambler=Y.SCRAMBLER_OWEN)
    with pytest.raises(Y.YartError, match="UNSUPPORTED"):
        Y.Context(light_sampler=Y.LIGHT_SAMPLER_UNIFORM)


def test_render_is_deterministic_and_capacity_independent():
    path = os.path.join(H.GOLDEN, "render_zoo.npz")
    _, d1, hdr1, ldr1, _ = PC.render_golden(path)
    _, d2, hdr2, ldr2, _ = PC.render_golden(path)
    assert H.bits_equal(hdr1, hdr2).all() and d1["total_rays"] == d2["total_rays"]
    g = PC.load(path)
    name, kw = PC.scene_from_golden(g)
    w, h, spp, first, mx, depth = (int(v) for v in g["settings"])
    cam = H.scene_camera(name)
    sc = Y.Scene(H.scene_file(name))
    c = Y.make_camera(w, h, cam["focal"], cam["fnum"], cam["pos"], cam["target"], (0, 0, 0), cam["exposure"])
    ctx = Y.Context(max_depth=depth, max_paths=4096)
    ctx.upload_scene(sc)
    ctx.set_camera(c)
    ctx.begin_frame(w, h, spp, 64, (0, 0, 0), Y.TONEMAP_AGX)
    ctx.render_wave(0, spp, 0)
    hdr3, _, st = ctx.resolve()
    assert H.bits_equal(hdr1, hdr3).all() and st.raysReference == d1["total_rays"]


def test_tile_shards_sum_to_full_frame_bitwise():
    path = os.path.join(H.GOLDEN, "render_cornell.npz")
    parts = [PC.render_golden(path, shard_index=k, shard_count=4, tile_size=16) for k in range(4)]
    hdr = sum(p[2] for p in parts)
    _, d1, hdr1, _, _ = PC.render_golden(path, tile_size=16)
    assert H.bits_equal(hdr, hdr1).all()
    assert sum(p[1]["total_rays"] for p in parts) == d1["total_rays"]


@pytest.fixture(scope="module")
def soup_100k():
    sc = Y.Scene(H.scene_file("soup", n_tris=100_000))
    ctx = Y.Context(max_depth=1)
    ctx.upload_scene(sc)
    return sc, ctx


def test_full_hd_primary_rays_device_trace_properties(soup_100k):
    """1920x1080 primary rays generated on the device, traced device-resident (the C2 microbench
    path): closest-hit must agree with the host-buffer hook on a sample, and an any-hit ray cut at
    the closest t + margin must be occluded, at t - margin unoccluded (where the hit is not grazing)."""
    sc, ctx = soup_100k
    cam = H.scene_camera("soup")
    W, Hh = 1920, 1080
    ctx.set_camera(Y.make_camera(W, Hh, cam["focal"], cam["fnum"], cam["pos"], cam["target"]))
    ctx.begin_frame(W, Hh, 16, 64, (0, 0, 0), Y.TONEMAP_NONE)
    n = W * Hh
    rays_dev, hits_dev = ctx.device_alloc(n * 32), ctx.device_alloc(n * 20)
    ctx.generate_primary_rays(0, 1, rays_dev)
    ms = ctx.trace_device(rays_dev, n, hits_dev, Y.TRACE_CLOSEST, repeat=2)
    assert ms > 0
    rays = np.empty((n, 8), np.float32)
    hits = np.empty(n, Y.COMPACT_HIT_DTYPE)
    ctx.d2h(rays, rays_dev)
    ctx.d2h(hits, hits_dev)
    ctx.device_free(rays_dev)
    ctx.device_free(hits_dev)
    assert np.allclose(np.linalg.norm(rays[:, 4:7], axis=1), 1.0, atol=1e-5)
    hit = hits["node"] >= 0
    assert 0.3 < hit.mean() < 1.0
    assert np.isinf(hits["t"][~hit]).all() and (hits["t"][hit] > 0.001).all()
    sel = np.random.default_rng(0).choice(n, 20000, replace=False)
    full, _ = ctx.trace(rays[sel], Y.TRACE_CLOSEST)
    assert np.array_equal(full["didHit"] == 1, hit[sel])
    assert np.array_equal(full["prim"][hit[sel]], hits["prim"][sel][hit[sel]])
    assert np.array_equal(full["t"].view(np.uint32), hits["t"][sel].view(np.uint32))
    hs = sel[hit[sel]]
    r_in = rays[hs].copy()
    r_in[:, 7] = hits["t"][hs] * (1 + 1e-4) + 1e-3
    occ, _ = ctx.trace(r_in, Y.TRACE_ANY)
    assert (occ["didHit"] == 1).all()
    r_out = rays[hs].copy()
    r_out[:, 7] = hits["t"][hs] * (1 - 1e-4) - 1e-3
    free, _ = ctx.trace(r_out, Y.TRACE_ANY)
    assert (free["didHit"] == 0).all()


def test_full_hd_render_wave_split_invariance(soup_100k):
    """1080p, primary + shadow only (C2 shape): 4 spp in one wave of 4 must produce the same
    per-sample radiance sums as the CPU-checked small case does — checked through the estimator-free
    property that a MEAN-estimator render is independent of how samples are grouped into chunks."""
    sc, _ = soup_100k
    cam = H.scene_camera("soup")
    W, Hh = 1920, 1080
    c = Y.make_camera(W, Hh, cam["focal"], cam["fnum"], cam["pos"], cam["target"])
    imgs = []
    for cap in (0, 3_000_000):  # default capacity (4 samples per chunk) vs 1 sample per chunk
        ctx = Y.Context(max_depth=1, max_paths=cap)
        ctx.upload_scene(sc)
        ctx.set_camera(c)
        ctx.begin_frame(W, Hh, 4, 64, (0, 0, 0), Y.TONEMAP_AGX, estimator=Y.ESTIMATOR_MEAN)
        ctx.render_wave(0, 4, 0)
        hdr, ldr, st = ctx.resolve()
        imgs.append((hdr, st.raysReference, st.raysExtend))
        assert st.raysExtend == W * Hh * 4
        ctx.close()
    assert H.bits_equal(imgs[0][0], imgs[1][0]).all() and imgs[0][1] == imgs[1][1]
    assert np.isfinite(imgs[0][0]).all() and imgs[0][0][..., :3].max() > 0


def test_empty_and_degenerate_inputs():
    ctx = Y.Context()
    sc = Y.Scene(H.scene_file("two_quads"))
    with pytest.raises(Y.YartError):
        ctx.trace(np.zeros((1, 8), np.float32))  # no scene yet
    ctx.upload_scene(sc)
    hits, _ = ctx.trace(np.zeros((0, 8), np.float32))
    assert len(hits) == 0
    # zero-direction / NaN / infinite-origin rays must neither hang nor crash
    bad = np.zeros((3, 8), np.float32)
    bad[1, 4:7] = np.nan
    bad[2, 0:3] = np.inf
    bad[:, 7] = np.inf
    hits, _ = ctx.trace(bad)
    assert hits["didHit"].tolist() == [0, 1, 0]  # what the reference does too: a NaN t passes `t <= tMin || hit.t <= t`


# ------------------------------------------------------------------------------------------
# BASELINE.json configs at (or near) full size
# ------------------------------------------------------------------------------------------
def _render_ctx(sc, cam, w, h, spp, waves, max_depth=30, tonemap=Y.TONEMAP_AGX, traversal=None, **frame_kw):
    c = Y.make_camera(w, h, cam["focal"], cam["fnum"], cam["pos"], cam["target"], (0, 0, 0), cam["exposure"])
    ctx = Y.Context(max_depth=max_depth, traversal=traversal)
    ctx.upload_scene(sc)
    ctx.set_camera(c)
    ctx.begin_frame(w, h, spp, 64, (0, 0, 0), tonemap, **frame_kw)
    taken = 0
    for wv in waves:
        ctx.render_wave(taken, wv, taken)
        taken += wv
    hdr, ldr, st = ctx.resolve()
    ctx.close()
    return hdr, ldr, st


C1 = dict(scene="cornell", kw={}, w=512, h=512, spp=16, max_depth=30)
C2 = dict(scene="soup", kw=dict(n_tris=1_000_000), w=1920, h=1080, spp=1, max_depth=1)
C3 = dict(scene="sponza", kw=dict(n_tris=260_000, tex_res=256, env_res=512), w=1920, h=1080, spp=1, max_depth=30)
C4 = dict(scene="mclaren", kw=dict(n_tris=2_000_000, env_res=512), w=1920, h=1080, spp=1, max_depth=30)
C5 = dict(scene="two_quads", kw={}, w=3840, h=2160, spp=30, waves=[15, 15], max_depth=2)


def render_config(cfg, traversal=None):
    """A BASELINE.json configuration rendered with the reference-order walk (or `traversal`): (scene, hdr, ldr, stats)."""
    sc = Y.Scene(H.scene_file(cfg["scene"], **cfg["kw"]))
    cam = H.scene_camera(cfg["scene"], **cfg["kw"])
    hdr, ldr, st = _render_ctx(sc, cam, cfg["w"], cfg["h"], cfg["spp"], cfg.get("waves", [cfg["spp"]]), max_depth=cfg["max_depth"],
                               traversal=traversal)
    return sc, hdr, ldr, st


def c2_primary_rays(sc):
    """Every 20th primary ray of the C2 frame, as the library generates them."""
    W, Hh, cam = C2["w"], C2["h"], H.scene_camera("soup")
    ctx = Y.Context(max_depth=1, traversal=Y.TRAVERSAL_AUTO)
    ctx.upload_scene(sc)
    ctx.set_camera(Y.make_camera(W, Hh, cam["focal"], cam["fnum"], cam["pos"], cam["target"]))
    ctx.begin_frame(W, Hh, 1, 64, (0, 0, 0), Y.TONEMAP_NONE)
    n = W * Hh
    rays_dev = ctx.device_alloc(n * 32)
    ctx.generate_primary_rays(0, 1, rays_dev)
    rays = np.empty((n, 8), np.float32)
    ctx.d2h(rays, rays_dev)
    ctx.device_free(rays_dev)
    return ctx, rays[::20].copy()


def hit_digests(hits):
    """What the reference's hit records pin: hit or miss, and the distance and triangle of every hit."""
    m = hits["didHit"] == 1
    return {"did_hit": H.digest(hits["didHit"]), "t": H.digest(hits["t"][m]), "prim": H.digest(hits["prim"][m])}


def _check_frame_recorded(tag, key, hdr, ldr, st):
    """The reference-order walk's frames and ray count against the reference's (recorded), bit for bit."""
    ref = H.recorded(key)
    assert st.raysReference == ref["rays"], f"{tag}: rays {st.raysReference} vs {ref['rays']}"
    assert H.digest(hdr) == ref["hdr"], f"{tag}: HDR differs from the reference's"
    assert H.digest(ldr) == ref["ldr"], f"{tag}: LDR differs from the reference's"


def test_c1_cornell_512_16spp_matches_reference_run_here():
    """configs[0] exactly: Cornell box, 512x512, 16 spp MIS+NEE, against the reference's frame."""
    _, hdr, ldr, st = render_config(C1)
    _check_frame_recorded("C1", "c1_cornell_512_16spp", hdr, ldr, st)


def test_c3_sponza_shape_1080p_matches_reference_run_here():
    """configs[2] shape at full resolution and triangle count (260 K tris, textured PBR + normal maps +
    alpha cut-outs, env light only), 1 spp."""
    sc, hdr, ldr, st = render_config(C3)
    assert 200_000 < sc.n_tris < 300_000
    _check_frame_recorded("C3", "c3_sponza_1080p_1spp", hdr, ldr, st)


def _check_wide_frame(tag, ref, hdr, ldr, st):
    """The wide walk's frame against the reference's: the north-star bars (relMSE < 1e-3 on the HDR frame and after
    AgX, ray counts), and pixels differing only where a path met a last-bit tie or a box-boundary hit — same
    triangles, same triangle arithmetic, different box culling (wide_bvh.cuh)."""
    rh, rl = H.rel_mse(hdr, ref["hdr"]), H.rel_mse(ldr, ref["ldr"])
    assert rh < 1e-3 and rl < 1e-3, f"{tag}: relMSE hdr {rh} ldr {rl}"
    assert abs(int(st.raysReference) - int(ref["rays"])) <= 1e-4 * ref["rays"], f"{tag}: rays {st.raysReference} vs {ref['rays']}"
    same = H.bits_equal(hdr, ref["hdr"]).all(-1).mean()
    print(f"{tag} wide: relMSE hdr {rh:.3g} ldr {rl:.3g}, {same:.7f} of the pixels bit-identical, rays {st.raysReference} vs {ref['rays']}")
    assert same > 0.999, f"{tag}: only {same} of the pixels are bit-identical to the reference"


def test_c2_soup_1m_tris_1080p_matches_reference_run_here():
    """configs[1] EXACTLY as bench.py times it (1 M-triangle soup, 1920x1080, primary + shadow rays, maxDepth 1),
    1 spp, against the reference's frame and ray count, then hit records of 100 K of the frame's primary rays against
    RayIntegrator::testNode.  The reference-order walk reproduces the reference bit for bit (checked against the
    recorded digests first), so its frame and hits then stand for the reference's in the checks of the wide walk."""
    sc, hdr, ldr, st = render_config(C2)
    assert sc.n_tris == 1_000_002  # the soup + the two triangles of the light quad
    _check_frame_recorded("C2", "c2_soup_1080p_1spp", hdr, ldr, st)
    ref = dict(hdr=hdr, ldr=ldr, rays=int(st.raysReference))
    _, hdr, ldr, st = render_config(C2, traversal=Y.TRAVERSAL_WIDE)  # what bench.py times
    _check_wide_frame("C2", ref, hdr, ldr, st)
    # ray level: the same frame's primary rays, every 20th, closest hit + any hit, both walks
    ctx, sel = c2_primary_rays(sc)
    rec = H.recorded("c2_soup_hits")
    assert H.digest(sel) == rec["rays"], "C2: the primary rays differ from those the reference traced"
    want, _ = ctx.trace(sel, Y.TRACE_CLOSEST | Y.TRACE_REFERENCE_ORDER)
    assert hit_digests(want) == rec["closest"], "C2: closest hits of the reference-order walk differ from the reference's"
    m = want["didHit"] == 1
    for walk in (Y.TRACE_REFERENCE_ORDER, Y.TRACE_WIDE):
        got, _ = ctx.trace(sel, Y.TRACE_CLOSEST | walk)
        assert np.array_equal(got["didHit"], want["didHit"])
        assert (np.abs(got["t"][m] - want["t"][m]) <= 1e-5 * np.abs(want["t"][m])).all()
        assert np.array_equal(got["t"][m].view(np.uint32), want["t"][m].view(np.uint32))
        ties = m & (got["prim"] != want["prim"])
        assert ties.sum() == 0 if walk == Y.TRACE_REFERENCE_ORDER else ties.sum() <= 4, f"C2: {ties.sum()} hit ids differ"
    sel[:, 7] = np.where(m, want["t"] * 0.5, 1e30)
    want_any, _ = ctx.trace(sel, Y.TRACE_ANY | Y.TRACE_REFERENCE_ORDER)
    assert H.digest(want_any["didHit"]) == rec["any"], "C2: any-hit results of the reference-order walk differ from the reference's"
    for walk in (Y.TRACE_REFERENCE_ORDER, Y.TRACE_WIDE):
        got_any, _ = ctx.trace(sel, Y.TRACE_ANY | walk)
        assert np.array_equal(got_any["didHit"], want_any["didHit"])
    ctx.close()


def test_c4_mclaren_shape_2m_tris_1080p_matches_reference_run_here():
    """configs[3] shape at full size (≈ 2 M tris, clearcoat / chrome / thin + solid glass with volume, emissive
    lamps + env), 1920x1080, full MIS+NEE paths, 1 spp, against the reference's frame (the reference-order walk's
    frame stands for it once it matches the recorded digests); plus determinism and tile shards summing to the full
    frame."""
    sc, *a = render_config(C4)
    assert sc.n_tris > 1_800_000
    _check_frame_recorded("C4", "c4_mclaren_1080p_1spp", *a)
    ref = dict(hdr=a[0], ldr=a[1], rays=int(a[2].raysReference))
    cam, w, h = H.scene_camera("mclaren", **C4["kw"]), C4["w"], C4["h"]
    wide = _render_ctx(sc, cam, w, h, 1, [1], traversal=Y.TRAVERSAL_WIDE)
    _check_wide_frame("C4", ref, *wide)
    b = _render_ctx(sc, cam, w, h, 1, [1])
    assert H.bits_equal(a[0], b[0]).all() and a[2].raysReference == b[2].raysReference
    assert np.isfinite(a[0]).all() and a[0][..., :3].mean() > 0.01
    parts = [_render_ctx(sc, cam, w, h, 1, [1], shard_index=k, shard_count=2) for k in range(2)]
    assert H.bits_equal(parts[0][0] + parts[1][0], a[0]).all()
    assert parts[0][2].raysReference + parts[1][2].raysReference == a[2].raysReference


def test_c5_4k_gmon_waves_match_reference_run_here():
    """configs[4] shape: 3840x2160, progressive GMoN waves (15 + 15 samples: m = 3 buckets per wave, blended with
    finishTile's weights), against the reference's frame (a two-quad scene so the CPU reference finishes in seconds);
    the reference-order walk's frame stands for it in the check of the wide walk once it matches the recorded digests."""
    _, hdr, ldr, st = render_config(C5)
    _check_frame_recorded("C5", "c5_two_quads_4k_30spp", hdr, ldr, st)
    ref = dict(hdr=hdr, ldr=ldr, rays=int(st.raysReference))
    _, hdr, ldr, st = render_config(C5, traversal=Y.TRAVERSAL_WIDE)
    _check_wide_frame("C5", ref, hdr, ldr, st)


def test_c5_4k_progressive_gmon_sharded_equals_unsharded():
    """configs[4] shape: 3840x2160, progressive waves (8, 16) with GMoN, tile-sharded over 2 contexts;
    the summed frames must be bit-identical to the unsharded render."""
    sp, cam = H.scene_file("cornell"), H.scene_camera("cornell")
    sc = Y.Scene(sp)
    w, h = 3840, 2160
    full = _render_ctx(sc, cam, w, h, 24, [8, 16])
    parts = [_render_ctx(sc, cam, w, h, 24, [8, 16], shard_index=k, shard_count=2) for k in range(2)]
    assert H.bits_equal(parts[0][0] + parts[1][0], full[0]).all()
    assert H.bits_equal(parts[0][1] + parts[1][1], full[1]).all()
    assert parts[0][2].raysReference + parts[1][2].raysReference == full[2].raysReference
    assert np.isfinite(full[0]).all()


def test_bucket_shards_combine_to_the_unsharded_render_bitwise():
    """Sample sharding by estimator bucket (yc_accumulate_wave / yc_bucket_device_ptrs / yc_finalize_wave):
    three contexts stand in for three GPUs, their GMoN accumulation buffers are added as int32 (what the NCCL
    all-reduce does) and the finalized frames must be bit-identical to yc_render_wave's, wave after wave
    (zoo scene: every material class; 64 + 128 samples → m = 11 then 15 buckets)."""
    sp, cam = H.scene_file("material_zoo"), H.scene_camera("material_zoo")
    sc = Y.Scene(sp)
    w, h, waves, G = 160, 90, [64, 128], 3
    c = Y.make_camera(w, h, cam["focal"], cam["fnum"], cam["pos"], cam["target"], (0, 0, 0), cam["exposure"])

    def ctx_new():
        ctx = Y.Context(max_depth=6)
        ctx.upload_scene(sc)
        ctx.set_camera(c)
        ctx.begin_frame(w, h, sum(waves), 64, (0, 0, 0), Y.TONEMAP_AGX)
        return ctx

    ref = ctx_new()
    shards = [ctx_new() for _ in range(G)]
    taken = 0
    for wv in waves:
        ref.render_wave(taken, wv, taken)
        total = None
        for g, ctx in enumerate(shards):
            ctx.accumulate_wave(taken, wv, bucket_shard=g, bucket_shard_count=G)
            ptr, nbytes, _, _ = ctx.bucket_device_ptrs()
            acc = np.empty(nbytes // 4, np.int32)
            ctx.d2h(acc, ptr)
            total = acc if total is None else total + acc
        for ctx in shards:
            ptr, _, _, _ = ctx.bucket_device_ptrs()
            ctx.h2d(ptr, total)
            ctx.finalize_wave(wv, taken)
        taken += wv
    hdr0, ldr0, st0 = ref.resolve()
    rays = 0
    for ctx in shards:
        hdr, ldr, st = ctx.resolve()
        assert H.bits_equal(hdr, hdr0).all() and H.bits_equal(ldr, ldr0).all()
        rays += st.raysReference
    assert rays == st0.raysReference
    assert np.isfinite(hdr0).all() and hdr0[..., :3].mean() > 0


def test_traversal_stack_spill_path_gives_identical_hits_and_frames(soup_100k):
    """The persistent kernels keep 25 stack entries per lane in shared memory and spill deeper ones to global
    memory.  With 3 shared entries (YcOptions.reserved2[0]) nearly every push spills: closest-hit and any-hit
    records of 1080p primary rays and a full-path render must not change by a bit."""
    sc, ctx = soup_100k
    cam = H.scene_camera("soup")
    W, Hh = 1920, 1080
    c = Y.make_camera(W, Hh, cam["focal"], cam["fnum"], cam["pos"], cam["target"])
    n = W * Hh
    out = []
    for entries in (0, 3):
        cx = Y.Context(max_depth=4, sh_stack_entries=entries)
        cx.upload_scene(sc)
        cx.set_camera(c)
        cx.begin_frame(W, Hh, 1, 64, (0, 0, 0), Y.TONEMAP_NONE)
        rays_dev, hits_dev = cx.device_alloc(n * 32), cx.device_alloc(n * 20)
        cx.generate_primary_rays(0, 1, rays_dev)
        rec = []
        for mode in (Y.TRACE_CLOSEST, Y.TRACE_ANY):
            cx.trace_device(rays_dev, n, hits_dev, mode)
            hits = np.empty(n, Y.COMPACT_HIT_DTYPE)
            cx.d2h(hits, hits_dev)
            rec.append(hits.tobytes())
        cx.device_free(rays_dev)
        cx.device_free(hits_dev)
        cx.render_wave(0, 1, 0)
        hdr, _, st = cx.resolve()
        out.append((rec, hdr, st.raysReference))
        cx.close()
    assert out[0][0][0] == out[1][0][0] and out[0][0][1] == out[1][0][1]
    assert H.bits_equal(out[0][1], out[1][1]).all() and out[0][2] == out[1][2]

    # and against the reference on a scene with nested transforms, alpha-tested and NEE-transparent materials
    path = os.path.join(H.GOLDEN, "render_zoo.npz")
    g = PC.load(path)
    name, kw = PC.scene_from_golden(g)
    w, h, spp, first, mx, depth = (int(v) for v in g["settings"])
    zc = H.scene_camera(name)
    cx = Y.Context(max_depth=depth, sh_stack_entries=2)
    cx.upload_scene(Y.Scene(H.scene_file(name)))
    cx.set_camera(Y.make_camera(w, h, zc["focal"], zc["fnum"], zc["pos"], zc["target"], (0, 0, 0), zc["exposure"]))
    cx.begin_frame(w, h, spp, 64, (0, 0, 0), Y.TONEMAP_AGX)
    cx.render_wave(0, spp, 0)
    hdr, _, st = cx.resolve()
    assert H.bits_equal(hdr, g["hdr"]).all() and st.raysReference == int(g["rays"])


@pytest.mark.parametrize("scene,depth,cap", [("material_zoo", 12, 0), ("material_zoo", 12, 20_000), ("cornell", 8, 6_000)])
def test_waves_left_in_flight_equal_waves_waited_for(scene, depth, cap):
    """yc_render_wave_async: the next wave's chunks start while the previous wave's tails, bucket sums and finalize
    still run.  Progressive GMoN waves (deep paths → tail kernels on the side streams; small capacities → many chunks
    per wave) issued back to back must give the bits of the same waves rendered one at a time, also when a synchronous
    call (a sub-rectangle wave) is mixed in, and the statistics must agree."""
    cam = H.scene_camera(scene)
    sc = Y.Scene(H.scene_file(scene))
    w, h = 320, 180
    c = Y.make_camera(w, h, cam["focal"], cam["fnum"], cam["pos"], cam["target"], (0, 0, 0), cam["exposure"])
    waves = [2, 4, 8, 8, 2, 8]
    out = []
    for mode in ("sync", "async"):
        ctx = Y.Context(max_depth=depth, max_paths=cap, tail_threshold=2048)
        ctx.upload_scene(sc)
        ctx.set_camera(c)
        frames = []
        for rep in range(2):
            ctx.begin_frame(w, h, sum(waves) + 2, 32, (0, 0, 0), Y.TONEMAP_AGX)
            taken = 0
            for k, wv in enumerate(waves):
                (ctx.render_wave_async if mode == "async" else ctx.render_wave)(taken, wv, taken)
                taken += wv
                if k == 3:  # a synchronous partial wave in the middle: left and right halves, one sample more each
                    ctx.render_wave(taken, 1, taken, rect=(0, 0, 100, h))
                    ctx.render_wave(taken, 1, taken, rect=(100, 0, w - 100, h))
                    taken += 1
            if mode == "async":
                ctx.wave_sync()
            hdr, ldr, st = ctx.resolve()
            frames.append((hdr, ldr, st.raysReference, st.raysExtend, st.raysShadow))
        out.append(frames)
        ctx.close()
    for (a, b) in zip(out[0], out[1]):
        assert H.bits_equal(a[0], b[0]).all() and H.bits_equal(a[1], b[1]).all()
        assert a[2:] == b[2:]


def test_graft_entry_smoke_in_a_fresh_process():
    """__graft_entry__.smoke() as the driver runs it: its own process, the library's defaults (wide walk)."""
    import subprocess
    import sys
    r = subprocess.run([sys.executable, "-c", "import __graft_entry__ as g; g.smoke()"], cwd=H.ROOT, capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0, (r.stdout + r.stderr)[-3000:]
    assert "smoke: ok" in r.stdout
