"""Image decoders of the host layer (yart_b200/host/images.cpp) against the reference's own loaders.

The reference decodes glTF textures with stb_image (loadTexture, src/core/texture.hpp:62-90) and the environment map
with stbi_loadf (loadTextureHDR, src/core/texture.cpp:21-35).  Every fixture under tests/golden/images was decoded by
the reference (oracle/_ref/oracle_ref texload / hdrload; generate.py next to the fixtures) and the recorded bytes must be
reproduced EXACTLY: baseline and progressive JPEG at every chroma layout, restart intervals, partial MCUs; PNG at every
bit depth, palette, colour keys, Adam7; Radiance RLE / flat."""
import glob
import os

import numpy as np
import pytest

import harness as H
import yart_b200 as Y
from yart_b200 import scenes as S

pytestmark = pytest.mark.usefixtures("hostsim_lib")
IMAGES = os.path.join(H.GOLDEN, "images")
LDR = sorted(glob.glob(os.path.join(IMAGES, "*.jpg")) + glob.glob(os.path.join(IMAGES, "*.png")))
HDR = sorted(glob.glob(os.path.join(IMAGES, "*.hdr")))


def test_fixtures_are_present():
    assert len(LDR) >= 30 and len(HDR) >= 3


@pytest.mark.parametrize("path", LDR, ids=os.path.basename)
def test_decoded_bytes_equal_stb_image(path):
    want = np.load(path + ".expect.npy")
    got = Y.decode_texture(open(path, "rb").read(), S.NONCOLOR, [0, 1, 2, 3])
    assert got.shape == want.shape
    bad = np.argwhere((got != want).any(-1))
    assert len(bad) == 0, f"{os.path.basename(path)}: {len(bad)} pixels differ, first {bad[:5].tolist()}: got {got[tuple(bad[0])]} want {want[tuple(bad[0])]}"


@pytest.mark.parametrize("path", HDR, ids=os.path.basename)
def test_radiance_floats_equal_stbi_loadf(path):
    want = np.load(path + ".expect.npy")
    got = Y.load_hdr(path)
    assert got.shape == want.shape and np.array_equal(got.view(np.uint32), want.view(np.uint32))


@pytest.mark.parametrize("path", LDR[::3], ids=os.path.basename)
def test_srgb_channel_conversion_equals_the_reference(path):
    """The sRGB → gamma-2 channel conversion of loadTexture, against the reference's (tests/golden/reference_digests.json)."""
    got = Y.decode_texture(open(path, "rb").read(), S.SRGB, [1, 2])
    assert H.digest(got) == H.recorded(f"texload_{os.path.basename(path)}_{S.SRGB}_12")


@pytest.mark.skipif(not H.have_oracle(), reason="oracle/_ref/oracle_ref not present")
@pytest.mark.parametrize("path", LDR[::3], ids=os.path.basename)
def test_recorded_expectations_are_the_reference_run_now(path, tmp_path):
    """The committed .expect.npy files are what the reference yields today (guards against stale fixtures), and the
    sRGB → gamma-2 channel conversion of loadTexture agrees too."""
    import struct
    out = str(tmp_path / "o.bin")
    H.run_oracle("texload", path, 2, 4, "0,1,2,3", out)
    raw = open(out, "rb").read()
    w, h, _ = struct.unpack_from("<III", raw, 0)
    assert np.array_equal(np.frombuffer(raw, np.uint8, w * h * 4, 12).reshape(h, w, 4), np.load(path + ".expect.npy"))
    H.run_oracle("texload", path, 1, 2, "1,2", out)
    raw = open(out, "rb").read()
    want = np.frombuffer(raw, np.uint8, w * h * 2, 12).reshape(h, w, 2)
    assert np.array_equal(Y.decode_texture(open(path, "rb").read(), S.SRGB, [1, 2]), want)


def test_unsupported_and_corrupt_images_fail_cleanly():
    with pytest.raises(Y.YartError, match="unsupported image format"):
        Y.decode_texture(b"GIF89a" + b"\0" * 64, S.SRGB, [0])
    jpg = open(os.path.join(IMAGES, "jpeg_420_q60.jpg"), "rb").read()
    with pytest.raises(Y.YartError, match="JPEG"):
        Y.decode_texture(jpg[:2] + b"\xff\xc0\x00\x0b\x08\x00\x00\x00\x10\x01\x01\x11\x00", S.SRGB, [0])  # zero height
    with pytest.raises(Y.YartError, match="arithmetic"):
        Y.decode_texture(jpg[:2] + b"\xff\xc9\x00\x0b\x08\x00\x10\x00\x10\x01\x01\x11\x00", S.SRGB, [0])
    png = open(os.path.join(IMAGES, "png_rgb8.png"), "rb").read()
    with pytest.raises(Y.YartError):
        Y.decode_texture(png[:len(png) // 2] + png[-12:], S.SRGB, [0])
    # truncated entropy-coded data: stb keeps what it decoded; so does this decoder (no crash, right size)
    got = Y.decode_texture(jpg[: len(jpg) * 2 // 3], S.NONCOLOR, [0, 1, 2, 3])
    assert got.shape == (29, 37, 4)


def test_glb_with_jpeg_textures_loads(tmp_path):
    """A GLB whose material textures are JPEGs (the common case for real assets) loads and renders."""
    from yart_b200.glbwriter import GlbBuilder
    jpg = open(os.path.join(IMAGES, "jpeg_420_q60.jpg"), "rb").read()
    g = GlbBuilder()
    tex = g.texture(jpg)  # an image stored in a bufferView of the BIN chunk, whatever its container format
    g.material({"pbrMetallicRoughness": {"baseColorTexture": {"index": tex}}})
    pos = np.array([[-1, -1, 0], [1, -1, 0], [1, 1, 0], [-1, 1, 0]], np.float32)
    nrm = np.tile(np.array([[0, 0, 1]], np.float32), (4, 1))
    uv = np.array([[0, 0], [1, 0], [1, 1], [0, 1]], np.float32)
    g.mesh([{"attributes": {"POSITION": g.accessor(pos, "VEC3"), "NORMAL": g.accessor(nrm, "VEC3"), "TEXCOORD_0": g.accessor(uv, "VEC2")},
             "indices": g.accessor(np.array([0, 1, 2, 0, 2, 3], np.uint16), "SCALAR"), "material": 0}])
    g.node({"mesh": 0}, root=True)
    p = tmp_path / "jpeg.glb"
    p.write_bytes(g.tobytes())
    ysc = tmp_path / "jpeg.ysc"
    Y.glb_to_ysc(str(p), str(ysc))
    sc = S.Scene.read(str(ysc)) if hasattr(S.Scene, "read") else None
    assert Y.Scene(str(p)).n_tris == 2
    if sc is not None:
        want = np.load(os.path.join(IMAGES, "jpeg_420_q60.jpg.expect.npy"))
        assert sc.textures[0].data.shape[:2] == want.shape[:2]
