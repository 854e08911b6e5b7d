"""The oracle is pinned two ways (SURVEY §8c: the reference ships no tests or vectors):
1. oracle/_ref/oracle_ref IS the unmodified reference; the committed fixtures in tests/golden are
   its recorded outputs, and re-running it here must reproduce them bit for bit.
2. the known-answer values recorded by the survey (SURVEY.md Appendix C, produced by calling the
   reference's functions directly in a separate build) must come out of it as well."""
import os
import struct

import numpy as np
import pytest

import harness as H
import parity_common as PC

needs_oracle = pytest.mark.skipif(not H.have_oracle(), reason="oracle/_ref/oracle_ref not built (make -C oracle ref)")


def test_golden_fixtures_present():
    assert len(PC.golden_files("kat")) >= 19
    assert len(PC.golden_files("trace")) >= 4
    assert len(PC.golden_files("render")) >= 6
    assert len(PC.golden_files("bvh")) >= 3
    assert len(PC.golden_files("naive")) >= 3
    assert len(PC.golden_files("scrambler")) >= 4
    assert len(PC.golden_files("medianbvh")) >= 3
    assert len(PC.golden_files("sampler")) >= 4


@needs_oracle
@pytest.mark.parametrize("path", PC.golden_files("kat"), ids=os.path.basename)
def test_oracle_reproduces_kat(path):
    g = PC.load(path)
    scene = str(g["scene"])
    out = H.oracle_kat(str(g["kind"]), g["blob"].tobytes(), H.scene_file(scene) if scene else None)
    assert H.bits_equal(out, g["out"]).all()


@needs_oracle
@pytest.mark.parametrize("path", PC.golden_files("variantkat"), ids=os.path.basename)
def test_oracle_reproduces_variant_kat(path):
    g = PC.load(path)
    out = H.oracle_kat(str(g["kind"]), g["blob"].tobytes(), H.scene_file(str(g["scene"])))
    assert H.bits_equal(out, g["out"]).all()


@needs_oracle
@pytest.mark.parametrize("path", PC.golden_files("trace"), ids=os.path.basename)
def test_oracle_reproduces_trace(path):
    g = PC.load(path)
    name, kw = PC.scene_from_golden(g)
    sp = H.scene_file(name, **kw)
    assert H.oracle_trace(sp, g["rays"], "closest").tobytes() == g["closest"].tobytes()
    assert H.oracle_trace(sp, g["rays"], "any").tobytes() == g["anyhit"].tobytes()


@needs_oracle
@pytest.mark.parametrize("path", PC.golden_files("render")[:3], ids=os.path.basename)
def test_oracle_reproduces_render_any_thread_count(path):
    g = PC.load(path)
    name, kw = PC.scene_from_golden(g)
    w, h, spp, first, mx, depth = (int(v) for v in g["settings"])
    r = H.oracle_render(H.scene_file(name, **kw), w, h, spp, H.scene_camera(name, **kw), first=first, max=mx,
                        maxdepth=depth, tonemap=str(g["tonemap"]), threads=2)
    assert r["rays"] == int(g["rays"])
    assert H.bits_equal(r["hdr"], g["hdr"]).all() and H.bits_equal(r["ldr"], g["ldr"]).all()


@needs_oracle
@pytest.mark.parametrize("path", PC.golden_files("naive"), ids=os.path.basename)
def test_oracle_reproduces_naive_render(path):
    g = PC.load(path)
    name, kw = PC.scene_from_golden(g)
    w, h, spp, first, mx, depth = (int(v) for v in g["settings"])
    r = H.oracle_render(H.scene_file(name, **kw), w, h, spp, H.scene_camera(name, **kw), first=first, max=mx,
                        maxdepth=depth, tonemap=str(g["tonemap"]), threads=2, integrator="naive")
    assert r["rays"] == int(g["rays"])
    assert H.bits_equal(r["hdr"], g["hdr"]).all() and H.bits_equal(r["ldr"], g["ldr"]).all()


@needs_oracle
@pytest.mark.parametrize("path", PC.golden_files("scrambler"), ids=os.path.basename)
def test_oracle_reproduces_scrambler_render(path):
    g = PC.load(path)
    name, kw = PC.scene_from_golden(g)
    w, h, spp, first, mx, depth = (int(v) for v in g["settings"])
    r = H.oracle_render(H.scene_file(name, **kw), w, h, spp, H.scene_camera(name, **kw), first=first, max=mx,
                        maxdepth=depth, tonemap=str(g["tonemap"]), threads=2, scrambler=str(g["scrambler"]))
    assert r["rays"] == int(g["rays"])
    assert H.bits_equal(r["hdr"], g["hdr"]).all() and H.bits_equal(r["ldr"], g["ldr"]).all()


@needs_oracle
@pytest.mark.parametrize("path", PC.golden_files("sampler"), ids=os.path.basename)
def test_oracle_reproduces_rng_sampler_render(path):
    g = PC.load(path)
    name, kw = PC.scene_from_golden(g)
    w, h, spp, first, mx, depth = (int(v) for v in g["settings"])
    r = H.oracle_render(H.scene_file(name, **kw), w, h, spp, H.scene_camera(name, **kw), first=first, max=mx,
                        maxdepth=depth, tonemap=str(g["tonemap"]), threads=2, sampler=str(g["sampler"]))
    assert r["rays"] == int(g["rays"])
    assert H.bits_equal(r["hdr"], g["hdr"]).all() and H.bits_equal(r["ldr"], g["ldr"]).all()


@needs_oracle
def test_survey_appendix_c_sampler_vectors():
    # SURVEY.md Appendix C: startPixelSample(px, s) then get2D, get2D, get1D, get1D
    cases = [
        (16, (3, 5), 0, [0.102555193, 0.584350109, 0.148540556, 0.324390888, 0.855917573, 0.421969295]),
        (16, (3, 5), 1, [0.318425208, 0.0620214753, 0.36125052, 0.840532362, 0.0274253599, 0.0999764204]),
        (16, (3, 5), 7, [0.247990549, 0.85945183, 0.594547987, 0.883081615, 0.918124795, 0.293590724]),
        (1024, (3, 5), 0, [0.600305319, 0.143533796, 0.431639761, 0.926101685, 0.420363069, 0.0162910819]),
        (1024, (3, 5), 7, [0.327253789, 0.245098159, 0.135244325, 0.10426487, 0.198218539, 0.80921936]),
    ]
    for spp, (x, y), s, want in cases:
        blob = struct.pack("<II3I", spp, 1, x, y, s)
        out = H.oracle_kat("sampler", blob)
        assert np.array_equal(out[:6], np.array(want, np.float32)), (spp, x, y, s, out[:6])


@needs_oracle
def test_survey_appendix_c_function_vectors():
    # ggxE(0.5,0.5), ggxEavg(0.5), ggxBaseE(0.04,0.5,0.3), ggxBaseEavg(0.04,0.5) and the UB cases
    out = H.oracle_kat("lut", struct.pack("<I4f", 1, 0.5, 0.5, 0.3, 1.5))
    assert out[0] == np.float32(0.857923031) and out[1] == np.float32(0.882156849)
    out = H.oracle_kat("lut", struct.pack("<I4f", 1, 0.04, 0.5, 0.3, 1.5))
    assert out[2] == np.float32(0.117981426) and out[3] == np.float32(0.0795770735)
    out = H.oracle_kat("lut", struct.pack("<I4f", 1, -0.5, 0.5, -0.3, 1.5))
    assert abs(out[0] - 0.825075) < 1e-6
    out = H.oracle_kat("lut", struct.pack("<I4f", 1, 0.04, 0.5, -0.3, 1.5))
    assert abs(out[2] - 0.0622205) < 1e-7
    # AgX[look none](0.18) and (2, 0.5, 0.1)
    out = H.oracle_kat("agx", struct.pack("<II6f", 0, 2, 0.18, 0.18, 0.18, 2.0, 0.5, 0.1))
    want = np.array([0.214467093, 0.214532301, 0.214536577, 0.807287812, 0.449624062, 0.21069032], np.float32)
    assert np.array_equal(out, want)
    # GMoNEstimator(16,15) fed s_i = (i%5, 0.5*(i%3), i==7 ? 100 : 1)
    s = np.array([[i % 5, 0.5 * (i % 3), 100.0 if i == 7 else 1.0] for i in range(16)], np.float32)
    out = H.oracle_kat("gmon", struct.pack("<II", 16, 1) + s.tobytes())
    assert np.array_equal(out[:3], np.array([1.88888884, 0.5, 7.5999999], np.float32))


@needs_oracle
def test_recorded_digests_are_the_reference_run_now(hostsim_lib):
    """tests/golden/reference_digests.json, which the parity tests compare with, is what the reference computes today
    for their inputs (tests/golden/record_digests.py)."""
    import json
    import sys
    sys.path.insert(0, H.GOLDEN)
    import record_digests
    with open(H.REFERENCE_DIGESTS) as f:
        want = json.load(f)
    got = record_digests.reference_outputs()
    assert sorted(got) == sorted(want)
    assert [k for k in sorted(want) if got[k] != want[k]] == []
