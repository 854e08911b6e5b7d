"""Randomised scenes against the reference's frames (recorded in tests/golden/reference_digests.json): every material
feature, nested / non-uniform transforms, degenerate triangles, all light types, DOF with disk and polygon apertures,
non-power-of-two sample counts, progressive waves, background colour — whole frames must match bit for bit.
CPU: the hostsim build.  GPU (`-m gpu`): the CUDA library."""
import numpy as np
import pytest

import harness as H
import yart_b200 as Y
from yart_b200 import scenes

TONEMAPS = ["agx", "golden", "punchy", "none"]
TM = {"none": Y.TONEMAP_NONE, "agx": Y.TONEMAP_AGX, "golden": Y.TONEMAP_AGX_GOLDEN, "punchy": Y.TONEMAP_AGX_PUNCHY}


def case_settings(seed):
    """Scene file, camera and render settings of random scene `seed`."""
    cam = scenes.random_scene(seed).camera
    spp = cam["spp"]
    first, mx = (spp, spp) if seed % 3 else (1, max(2, spp // 2))
    return dict(path=H.scene_file("random_scene", seed=seed), cam=cam, w=cam["w"], h=cam["h"], spp=spp, first=first, max=mx,
                bg=(0.0, 0.0, 0.0) if seed % 2 else (0.1, 0.2, 0.3), tonemap=TONEMAPS[seed % 4], depth=30 if seed % 5 else 3,
                tile=16 if seed % 2 else 64)


def render_case(seed, integrator="mis", scrambler="fastowen", sampler="sobol", traversal=None):
    """Renders random scene `seed` with the active library (and `traversal`, if given): (render data, hdr, ldr)."""
    k = case_settings(seed)
    cam, w, h = k["cam"], k["w"], k["h"]
    s = Y.Scene(k["path"])
    c = Y.make_camera(w, h, cam["focal"], cam["fnum"], cam["pos"], cam["target"], (0, 0, 0), cam["exposure"], cam["sides"])
    r = Y.Renderer(w, h, c, s, samples=k["spp"], first_wave_samples=k["first"], max_wave_samples=k["max"], max_depth=k["depth"],
                   background=k["bg"], tonemap=TM[k["tonemap"]], tile_size=k["tile"],
                   integrator=Y.INTEGRATOR_NAIVE if integrator == "naive" else Y.INTEGRATOR_MIS,
                   scrambler={"fastowen": Y.SCRAMBLER_FAST_OWEN, "owen": Y.SCRAMBLER_OWEN, "binary": Y.SCRAMBLER_BINARY_PERMUTE}[scrambler],
                   sampler={"sobol": Y.SAMPLER_SOBOL, "naive": Y.SAMPLER_NAIVE, "stratified": Y.SAMPLER_STRATIFIED}[sampler],
                   traversal=traversal)
    d = r.render_sync()
    hdr, ldr, _ = r.read()
    r.close()
    return d, hdr, ldr


def run_case(seed, integrator="mis", scrambler="fastowen", sampler="sobol"):
    d, hdr, ldr = render_case(seed, integrator, scrambler, sampler)
    ref = H.recorded(f"random_scene_{seed}")
    assert d["total_rays"] == ref["rays"], f"seed {seed}: rays {d['total_rays']} vs {ref['rays']}"
    assert H.digest(hdr) == ref["hdr"], f"seed {seed}: HDR differs from the reference's"
    assert H.digest(ldr) == ref["ldr"], f"seed {seed}: LDR differs from the reference's"
    assert np.isfinite(hdr[..., :3]).any()


@pytest.mark.parametrize("seed", range(16))
def test_random_scene_bit_exact_hostsim(seed, hostsim_lib):
    run_case(seed)


@pytest.mark.gpu
@pytest.mark.parametrize("seed", range(16, 40))
def test_random_scene_bit_exact_cuda(seed, cuda_lib):
    run_case(seed)


@pytest.mark.parametrize("seed", range(100, 106))
def test_random_scene_naive_integrator_bit_exact_hostsim(seed, hostsim_lib):
    run_case(seed, "naive")


@pytest.mark.gpu
@pytest.mark.parametrize("seed", range(106, 114))
def test_random_scene_naive_integrator_bit_exact_cuda(seed, cuda_lib):
    run_case(seed, "naive")


@pytest.mark.parametrize("seed", range(200, 206))
def test_random_scene_other_scramblers_bit_exact_hostsim(seed, hostsim_lib):
    run_case(seed, scrambler="owen" if seed % 2 else "binary")


@pytest.mark.gpu
@pytest.mark.parametrize("seed", range(206, 214))
def test_random_scene_other_scramblers_bit_exact_cuda(seed, cuda_samplers_lib):
    run_case(seed, scrambler="owen" if seed % 2 else "binary")


@pytest.mark.parametrize("seed", range(300, 306))
def test_random_scene_rng_samplers_bit_exact_hostsim(seed, hostsim_lib):
    run_case(seed, sampler="naive" if seed % 2 else "stratified")


@pytest.mark.gpu
@pytest.mark.parametrize("seed", range(306, 314))
def test_random_scene_rng_samplers_bit_exact_cuda(seed, cuda_samplers_lib):
    run_case(seed, sampler="naive" if seed % 2 else "stratified")
