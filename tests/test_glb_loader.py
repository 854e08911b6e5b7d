"""SURVEY §8f rank 1/3: the from-scratch GLB reader (host/glb.cpp ↔ src/gltf/gltf.cpp) and the PPM writer.

The reference's loader cannot be built here (fastgltf is not vendored), so the reader is pinned by
(i) texture decode + conversion against the reference's own loadTexture (stb_image + glibc pow, through
`oracle_ref texload`; recorded in tests/golden/reference_digests.json), (ii) an independently constructed expected
scene (.ysc bytes) for a GLB that exercises every branch of gltf.cpp, and (iii) rendering the loaded scene against the
reference's recorded frame."""
import os

import numpy as np
import pytest

import harness as H
import yart_b200 as Y
from yart_b200 import scenes as S
from yart_b200.glbwriter import GlbBuilder, png_encode

pytestmark = pytest.mark.usefixtures("hostsim_lib")
f32 = np.float32
TEXLOAD_CASES = ((S.SRGB, [0, 1, 2, 3]), (S.NONCOLOR, [1, 2]), (S.NONCOLOR, [0]), (S.SRGB, [0, 1, 2]), (S.LINEAR, [2, 1, 0]))


def texload_key(name: str, tex_type: int, channels) -> str:
    return f"texload_{name}_{tex_type}_{''.join(map(str, channels))}"


def reference_texload(name: str, png: bytes, tex_type: int, channels) -> np.ndarray:
    """loadTexture's result for the named test image: the product's decode, checked against the reference's."""
    got = Y.decode_texture(png, tex_type, channels)
    assert H.digest(got) == H.recorded(texload_key(name, tex_type, channels)), (name, tex_type, channels)
    return got


def sample_images():
    rng = np.random.default_rng(3)
    grad = (np.add.outer(np.arange(13), np.arange(17)) * 7 % 256).astype(np.uint8)
    return {
        "rgba": rng.integers(0, 256, (9, 11, 4), dtype=np.uint8),
        "rgb": rng.integers(0, 256, (16, 8, 3), dtype=np.uint8),
        "grey": grad,
        "grey_alpha": np.stack([grad, 255 - grad], -1),
        "smooth_rgb": np.stack([grad, grad[::-1], grad[:, ::-1]], -1),  # filters actually predict something
    }


def sample_png(name: str) -> bytes:
    rng = np.random.default_rng(5)
    if name == "palette":
        pal = rng.integers(0, 256, (37, 3), dtype=np.uint8)
        png = png_encode(rng.integers(0, 37, (10, 12), dtype=np.uint8), palette=pal)
    elif name == "rgb16":
        png = png_encode(rng.integers(0, 65536, (7, 9, 3)).astype(np.uint16), bit_depth=16)
    else:
        png = png_encode(sample_images()[name])
    return png


@pytest.mark.parametrize("name", ["rgba", "rgb", "grey", "grey_alpha", "smooth_rgb", "palette", "rgb16"])
def test_png_decode_and_conversion_match_reference_loadTexture(name):
    png = sample_png(name)
    for tex_type, channels in TEXLOAD_CASES:
        reference_texload(name, png, tex_type, channels)


def test_png_errors():
    with pytest.raises(Y.YartError, match="JPEG"):
        Y.decode_texture(b"\xff\xd8\xff\xe0" + b"\0" * 64, S.SRGB, [0, 1, 2, 3])
    with pytest.raises(Y.YartError, match="unsupported image format"):
        Y.decode_texture(b"GIF89a" + b"\0" * 64, S.SRGB, [0])
    good = png_encode(sample_images()["rgb"])
    with pytest.raises(Y.YartError, match="inflate"):
        Y.decode_texture(good[:len(good) // 2] + good[-12:], S.SRGB, [0])


# ---- float32 restatement of the loader's matrix arithmetic (gltf.cpp:6-18, 285-288; mat.hpp:262-273) ----
def mat_mul(a, b):
    r = np.zeros((4, 4), f32)
    for i in range(4):
        for j in range(4):
            s = f32(0)
            for k in range(4):
                s = f32(s + f32(a[i, k] * b[k, j]))
            r[i, j] = s
    return r


def trs_matrix(t, q, s):
    qi, qj, qk, qr = (f32(x) for x in q)
    h = f32(0.5)
    half = np.array([[h - (qj * qj + qk * qk), qi * qj - qr * qk, qi * qk + qr * qj, 0],
                     [qi * qj + qr * qk, h - (qi * qi + qk * qk), qj * qk - qr * qi, 0],
                     [qi * qk - qr * qj, qj * qk + qr * qi, h - (qi * qi + qj * qj), 0],
                     [0, 0, 0, h]], f32)
    rot = (half * f32(2)).astype(f32)
    T = np.eye(4, dtype=f32)
    T[:3, 3] = np.asarray(t, f32)
    Sm = np.diag(np.array([s[0], s[1], s[2], 1], f32)).astype(f32)
    return mat_mul(mat_mul(T, rot), Sm)


def quat(axis, deg):
    a = np.asarray(axis, np.float64)
    a = a / np.linalg.norm(a)
    h = np.deg2rad(deg) / 2
    return [float(f32(x)) for x in (*(a * np.sin(h)), np.cos(h))]


def build_case(tmp_path, check_textures=True):
    """A GLB touching every branch of gltf.cpp, plus the scene it must load as."""
    imgs = sample_images()
    g = GlbBuilder()
    png_base, png_mr, png_nrm, png_em = (png_encode(imgs[k]) for k in ("rgba", "rgb", "smooth_rgb", "rgb"))
    t_base, t_mr, t_nrm, t_em = g.texture(png_base), g.texture(png_mr), g.texture(png_nrm), g.texture(png_em)
    g.material({"pbrMetallicRoughness": {"baseColorFactor": [0.9, 0.8, 0.7, 1.0], "roughnessFactor": 0.6, "metallicFactor": 0.2,
                                         "baseColorTexture": {"index": t_base}, "metallicRoughnessTexture": {"index": t_mr}},
                "normalTexture": {"index": t_nrm, "scale": 0.7}})
    g.material({"emissiveFactor": [1.0, 0.5, 0.25], "emissiveTexture": {"index": t_em},
                "extensions": {"KHR_materials_emissive_strength": {"emissiveStrength": 12.0}}})
    g.material({"pbrMetallicRoughness": {"roughnessFactor": 0.05, "metallicFactor": 0.0},
                "extensions": {"KHR_materials_transmission": {"transmissionFactor": 0.9}, "KHR_materials_ior": {"ior": 1.33},
                               "KHR_materials_volume": {"attenuationColor": [0.5, 0.8, 0.9], "attenuationDistance": 2.0}}})
    g.material({"pbrMetallicRoughness": {"baseColorFactor": [0.1, 0.2, 0.8, 1.0], "roughnessFactor": 0.4},
                "extensions": {"KHR_materials_clearcoat": {"clearcoatFactor": 1.0, "clearcoatRoughnessFactor": 0.02},
                               "KHR_materials_anisotropy": {"anisotropyStrength": 0.6, "anisotropyRotation": 0.4}}})
    # mesh 0: two primitives (materials 0 and 3), the second with tangents; mesh 1: emissive quad; mesh 2: glass box
    b0 = S.MeshBuilder()
    b0.quad((-6, 0, 6), (6, 0, 6), (6, 0, -6), (-6, 0, -6), 0, uv_scale=2.0)
    b0.quad((-6, 0, -6), (6, 0, -6), (6, 7, -6), (-6, 7, -6), 0)
    m0a = b0.build()
    b1 = S.MeshBuilder()
    b1.box((-1, 0, -1), (1, 2, 1), 3)
    m0b = b1.build()
    bl = S.MeshBuilder()
    bl.quad((-1, 0, -1), (1, 0, -1), (1, 0, 1), (-1, 0, 1), 1)
    ml = bl.build()
    bg = S.MeshBuilder()
    bg.box((-0.8, 0, -0.8), (0.8, 1.6, 0.8), 2)
    mg = bg.build()

    def prim(m, mat, tangents, index_dtype):
        p, n, uv = g.interleaved(m.positions, m.normals, m.uvs)
        at = {"POSITION": p, "NORMAL": n, "TEXCOORD_0": uv}
        if tangents:
            at["TANGENT"] = g.accessor(m.tangents.astype(f32), "VEC4")
        idx = m.faces[:, :3].reshape(-1).astype(index_dtype)
        return {"attributes": at, "indices": g.accessor(idx, "SCALAR"), "material": mat, "mode": 4}
    mesh0 = g.mesh([prim(m0a, 0, False, np.uint16), prim(m0b, 3, True, np.uint8),
                    {"attributes": {"POSITION": 0}, "mode": 1}])  # a LINES primitive: skipped (gltf.cpp:197)
    mesh1 = g.mesh([prim(ml, 1, False, np.uint32)])
    mesh2 = g.mesh([prim(mg, 2, True, np.uint16)])
    # nodes: A(TRS) → B(rot, mesh0) ; C(translate, mesh1) ; D(translate+scale, mesh1 again) ; E(mesh2, default TRS)
    nB = g.node({"mesh": mesh0, "rotation": quat((0, 1, 0), 12.0)})
    trsA = dict(translation=[0.25, 0.0, -0.5], rotation=quat((0, 1, 0), -7.0), scale=[1.0, 1.0, 1.0])
    g.node({"children": [nB], **trsA}, root=True)
    trsC = dict(translation=[0.0, 6.5, 0.0])
    g.node({"mesh": mesh1, **trsC}, root=True)
    trsD = dict(translation=[3.0, 5.0, 1.0], scale=[0.5, 0.5, 0.5])
    g.node({"mesh": mesh1, **trsD}, root=True)
    g.node({"mesh": mesh2, "translation": [-2.5, 0.0, 1.0]}, root=True)
    glb = tmp_path / "case.glb"
    glb.write_bytes(g.tobytes())

    # ---- the scene gltf::load would build, constructed independently -------------------------------
    texload = reference_texload if check_textures else (lambda _, png, t, ch: Y.decode_texture(png, t, ch))
    e = S.Scene()
    e.textures = [S.Texture(texload("rgba", png_base, S.SRGB, [0, 1, 2, 3]), S.SRGB),
                  S.Texture(texload("rgb", png_mr, S.NONCOLOR, [1, 2]), S.NONCOLOR),
                  S.Texture(texload("smooth_rgb", png_nrm, S.NONCOLOR, [0, 1, 2]), S.NONCOLOR),
                  S.Texture(texload("rgb", png_em, S.SRGB, [0, 1, 2]), S.SRGB)]
    e.materials = [
        S.Material(base=(f32(0.9), f32(0.8), f32(0.7)), base_tex=0, mr_tex=1, normal_tex=2, roughness=0.6, metallic=0.2,
                   clearcoat_roughness=0.03, normal_scale=0.7, thin=1),
        S.Material(emis_tex=3, roughness=1.0, metallic=1.0, clearcoat_roughness=0.03, thin=1,
                   emission=tuple(float(f32(x) * f32(12.0)) for x in (1.0, 0.5, 0.25))),
        S.Material(roughness=0.05, metallic=0.0, transmission=0.9, ior=1.33, clearcoat_roughness=0.03, thin=1,
                   volume_color=(0.5, 0.8, 0.9), volume_density=float(f32(1.0) / f32(2.0))),
        S.Material(base=(0.1, 0.2, 0.8), roughness=0.4, metallic=1.0, clearcoat=1.0, clearcoat_roughness=0.02, anisotropic=0.6,
                   aniso_rotation=0.4, thin=1),
    ]
    zero_t = lambda m: np.zeros((len(m.positions), 4), f32)
    merged = S.Mesh(np.concatenate([m0a.positions, m0b.positions]), np.concatenate([m0a.normals, m0b.normals]),
                    np.concatenate([zero_t(m0a), m0b.tangents]), np.concatenate([m0a.uvs, m0b.uvs]),
                    np.concatenate([m0a.faces, m0b.faces + np.array([len(m0a.positions)] * 3 + [0], np.uint32)]))
    light_mesh = S.Mesh(ml.positions, ml.normals, zero_t(ml), ml.uvs, ml.faces)
    glass = S.Mesh(mg.positions, mg.normals, mg.tangents, mg.uvs, mg.faces)
    e.meshes = [merged, light_mesh, glass]
    ident = trs_matrix((0, 0, 0), (0, 0, 0, 1), (1, 1, 1))
    mA = trs_matrix(trsA["translation"], trsA["rotation"], trsA["scale"])
    mB = trs_matrix((0, 0, 0), quat((0, 1, 0), 12.0), (1, 1, 1))
    mC = trs_matrix(trsC["translation"], (0, 0, 0, 1), (1, 1, 1))
    mD = trs_matrix(trsD["translation"], (0, 0, 0, 1), trsD["scale"])
    mE = trs_matrix([-2.5, 0.0, 1.0], (0, 0, 0, 1), (1, 1, 1))
    assert np.array_equal(ident, np.eye(4, dtype=f32))
    e.nodes = [S.Node(-1, -1), S.Node(0, -1, mA), S.Node(1, 0, mB), S.Node(0, 1, mC), S.Node(0, 1, mD), S.Node(0, 2, mE)]
    em = e.materials[1].emission
    # one AreaLight per emissive triangle and node, transform = node.transform * globalTransform (identity parents)
    for m in (mC, mD):
        for tri in range(2):
            e.lights.append(S.Light(S.AREA, 1, tri, em, mat_mul(m, np.eye(4, dtype=f32))))
    light_mesh.light_idx[:] = [0, 1]  # sic: the per-node counter restarts (SURVEY Appendix A.21)
    return str(glb), e


def test_glb_loads_as_the_expected_scene(tmp_path):
    glb, expected = build_case(tmp_path)
    want, got = tmp_path / "want.ysc", tmp_path / "got.ysc"
    expected.write(str(want))
    Y.glb_to_ysc(glb, str(got))
    assert got.read_bytes() == want.read_bytes()


GLB_CAM = dict(pos=(0.5, 4.0, 14.0), target=(0.0, 2.5, 0.0), focal=35.0, fnum=0.0, exposure=0.0)


def glb_env():
    return S.sky_hdr(16, 16, 5, 50.0)


def render_glb_case(tmp_path):
    """The GLB case straight from the file, with a sky, 64x40 at 8 spp: (render data, hdr, ldr, PPM bytes)."""
    glb, _ = build_case(tmp_path, check_textures=False)
    cam = GLB_CAM
    sc = Y.Scene(glb, env=glb_env(), env_radius=80.0)
    assert sc.flat.nLights == 5 and sc.flat.nArea == 4 and sc.flat.nMeshes == 3
    c = Y.make_camera(64, 40, 35.0, 0.0, cam["pos"], cam["target"])
    r = Y.Renderer(64, 40, c, sc, samples=8, first_wave_samples=8, max_wave_samples=8)
    d = r.render_sync()
    hdr, ldr, _ = r.read()
    r.write_ppm(str(tmp_path / "ours.ppm"))
    r.close()
    return d, hdr, ldr, (tmp_path / "ours.ppm").read_bytes()


def test_glb_scene_renders_bit_exactly_like_the_reference(tmp_path):
    d, hdr, ldr, ppm = render_glb_case(tmp_path)
    ref = H.recorded("glb_scene_64x40_8spp")
    assert d["total_rays"] == ref["rays"]
    assert H.digest(hdr) == ref["hdr"] and H.digest(ldr) == ref["ldr"]
    # output::writePPM parity (ppm.cpp:6-21)
    assert H.digest(np.frombuffer(ppm, np.uint8)) == ref["ppm"]


def test_glb_errors(tmp_path):
    p = tmp_path / "x.glb"
    p.write_bytes(b"nope" + b"\0" * 32)
    with pytest.raises(Y.YartError, match="not a glTF file"):
        Y.Scene(str(p))
    glb, _ = build_case(tmp_path, check_textures=False)
    raw = open(glb, "rb").read()
    p.write_bytes(raw[: len(raw) - 100])
    with pytest.raises(Y.YartError, match="truncated"):
        Y.Scene(str(p))
    g = GlbBuilder()
    g.material({})
    pos = np.zeros((3, 3), f32)
    g.mesh([{"attributes": {"POSITION": g.accessor(pos, "VEC3")}, "indices": g.accessor(np.arange(3, dtype=np.uint16), "SCALAR")}])
    g.node({"mesh": 0}, root=True)
    p.write_bytes(g.tobytes())
    with pytest.raises(Y.YartError, match="NORMAL"):
        Y.Scene(str(p))
    with pytest.raises(Y.YartError):
        Y.Scene(str(tmp_path / "missing.glb"))


def test_hostile_sizes_are_rejected_not_trusted(tmp_path):
    """ADVICE r1: counts / offsets in a .glb or .ysc are attacker-controlled.  Wrapping sums, negative or non-finite JSON
    numbers, a short `matrix`, and counts larger than the file must produce an error code — not a heap overrun, not an
    exception escaping the C ABI."""
    import json
    import struct

    def glb(doc, bin_bytes=b"\0" * 64):
        js = json.dumps(doc).encode()
        js += b" " * (-len(js) % 4)
        body = struct.pack("<II", len(js), 0x4E4F534A) + js + struct.pack("<II", len(bin_bytes), 0x004E4942) + bin_bytes
        return struct.pack("<III", 0x46546C67, 2, 12 + len(body)) + body

    def base(acc_pos, acc_idx=None, node=None):
        return {"asset": {"version": "2.0"}, "buffers": [{"byteLength": 64}],
                "bufferViews": [{"buffer": 0, "byteOffset": 0, "byteLength": 64}],
                "accessors": [acc_pos, acc_idx or {"bufferView": 0, "componentType": 5125, "count": 3, "type": "SCALAR"}],
                "meshes": [{"primitives": [{"attributes": {"POSITION": 0}, "indices": 1}]}],
                "nodes": [node or {"mesh": 0}], "scenes": [{"nodes": [0]}], "scene": 0}

    pos = {"bufferView": 0, "componentType": 5126, "type": "VEC3"}
    cases = {
        "wrapping_count": base(dict(pos, count=2 ** 63)),
        "huge_count": base(dict(pos, count=1e30)),
        "negative_count": base(dict(pos, count=-4)),
        "wrapping_offset": base(dict(pos, count=1, byteOffset=2 ** 64 - 8)),
        "index_count_beyond_view": base(dict(pos, count=3), {"bufferView": 0, "componentType": 5125, "count": 2 ** 62, "type": "SCALAR"}),
        "short_matrix": base(dict(pos, count=3), node={"mesh": 0, "matrix": [1, 0, 0]}),
        "view_beyond_bin": dict(base(dict(pos, count=3)), bufferViews=[{"buffer": 0, "byteOffset": 60, "byteLength": 2 ** 40}]),
    }
    for name, doc in cases.items():
        p = tmp_path / f"{name}.glb"
        p.write_bytes(glb(doc))
        with pytest.raises(Y.YartError):
            Y.Scene(str(p))
    # .ysc: a texture count / mesh size far beyond the file
    for name, payload in (("ysc_textures", b"YSC1" + struct.pack("<I", 0xFFFFFFF0)),
                          ("ysc_mesh", b"YSC1" + struct.pack("<III", 0, 0, 1) + struct.pack("<II", 0xFFFFFFFF, 0xFFFFFFFF))):
        p = tmp_path / f"{name}.ysc"
        p.write_bytes(payload + b"\0" * 32)
        with pytest.raises(Y.YartError, match="exceeds the file"):
            Y.Scene(str(p))


def test_gltf_json_with_external_and_data_uri_buffers_equals_the_glb(tmp_path):
    """.gltf (JSON) with its geometry in a .bin next to it, or in a base64 data URI, loads to the same scene as the
    equivalent .glb (fastgltf Options::LoadExternalBuffers, gltf.cpp:335); images inside such buffers are dropped, as in
    the reference (gltf.cpp:33-41 accepts ByteView buffers only)."""
    import base64
    import json
    import struct
    g = GlbBuilder()
    g.material({"pbrMetallicRoughness": {"baseColorFactor": [0.2, 0.4, 0.6, 1.0], "roughnessFactor": 0.5}})
    b0 = S.MeshBuilder()
    b0.box((-1, 0, -1), (1, 2, 1), 0)
    m = b0.build()
    g.mesh([{"attributes": {"POSITION": g.accessor(m.positions.astype(f32), "VEC3"), "NORMAL": g.accessor(m.normals.astype(f32), "VEC3"),
                            "TEXCOORD_0": g.accessor(m.uvs.astype(f32), "VEC2")},
             "indices": g.accessor(m.faces[:, :3].astype(np.uint32).reshape(-1), "SCALAR"), "material": 0}])
    g.node({"mesh": 0, "translation": [0.5, 0.0, -2.0]}, root=True)
    glb = g.tobytes()
    (tmp_path / "a.glb").write_bytes(glb)
    jlen, = struct.unpack_from("<I", glb, 12)
    doc = json.loads(glb[20:20 + jlen])
    blen, = struct.unpack_from("<I", glb, 20 + jlen)
    bin_bytes = glb[28 + jlen: 28 + jlen + blen]
    ext = dict(doc, buffers=[{"byteLength": len(bin_bytes), "uri": "geometry.bin"}])
    (tmp_path / "geometry.bin").write_bytes(bin_bytes)
    (tmp_path / "ext.gltf").write_text(json.dumps(ext))
    emb = dict(doc, buffers=[{"byteLength": len(bin_bytes), "uri": "data:application/octet-stream;base64," + base64.b64encode(bin_bytes).decode()}])
    (tmp_path / "emb.gltf").write_text(json.dumps(emb))
    out = {}
    for name in ("a.glb", "ext.gltf", "emb.gltf"):
        Y.glb_to_ysc(str(tmp_path / name), str(tmp_path / (name + ".ysc")))
        out[name] = (tmp_path / (name + ".ysc")).read_bytes()
    assert out["a.glb"] == out["ext.gltf"] == out["emb.gltf"]
    with pytest.raises(Y.YartError, match="next to the asset"):
        (tmp_path / "bad.gltf").write_text(json.dumps(dict(doc, buffers=[{"byteLength": 4, "uri": "../secret.bin"}])))
        Y.Scene(str(tmp_path / "bad.gltf"))
    with pytest.raises(Y.YartError, match="cannot open external buffer"):
        (tmp_path / "missing.gltf").write_text(json.dumps(dict(doc, buffers=[{"byteLength": 4, "uri": "nope.bin"}])))
        Y.Scene(str(tmp_path / "missing.gltf"))
