"""Writes tests/golden/reference_digests.json: what the reference computes for the inputs of the parity tests that compare
whole frames, hit records or decoded textures with it, as digests (harness.digest) and ray counts, so that the suite
needs neither the reference sources nor oracle/_ref to run them.

Every value comes from the reference build (oracle/_ref/oracle_ref) run on the tests' inputs.  The product's CPU build
only makes inputs, as the tests always did: the C2 primary rays the reference traces, and the .ysc of the GLB case
(the reference's glTF loader cannot be built).  tests/test_oracle_golden.py::test_recorded_digests_are_the_reference_run_now
runs the same computation wherever oracle/_ref is built and compares it with the committed file.

    python tests/golden/record_digests.py        (needs oracle/_ref: make -C oracle ref)
"""
import json
import os
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path[:0] = [os.path.dirname(os.path.dirname(HERE)), os.path.dirname(HERE)]

import numpy as np  # noqa: E402

import harness as H  # noqa: E402
import yart_b200 as Y  # noqa: E402
import test_fuzz_parity as FZ  # noqa: E402
import test_glb_loader as GL  # noqa: E402
import test_gpu_parity as GP  # noqa: E402
import test_image_decoders as ID  # noqa: E402
from yart_b200 import scenes as S  # noqa: E402

# test_fuzz_parity: seed → the variant its test renders
FUZZ = ([(s, {}) for s in range(0, 40)] + [(s, dict(integrator="naive")) for s in range(100, 114)] +
        [(s, dict(scrambler="owen" if s % 2 else "binary")) for s in range(200, 214)] +
        [(s, dict(sampler="naive" if s % 2 else "stratified")) for s in range(300, 314)])
CONFIGS = (("c1_cornell_512_16spp", GP.C1), ("c2_soup_1080p_1spp", GP.C2), ("c3_sponza_1080p_1spp", GP.C3),
           ("c4_mclaren_1080p_1spp", GP.C4), ("c5_two_quads_4k_30spp", GP.C5))


def frame(ref):
    return {"rays": int(ref["rays"]), "hdr": H.digest(ref["hdr"]), "ldr": H.digest(ref["ldr"])}


def reference_outputs() -> dict:
    """Every entry of reference_digests.json, computed by oracle/_ref/oracle_ref.  The active library (the product's
    CPU build) makes the C2 rays and the GLB case's .ysc."""
    out = {}
    for seed, kw in FUZZ:
        k = FZ.case_settings(seed)
        out[f"random_scene_{seed}"] = frame(H.oracle_render(
            k["path"], k["w"], k["h"], k["spp"], k["cam"], first=k["first"], max=k["max"], maxdepth=k["depth"],
            tonemap=k["tonemap"], bg="%g,%g,%g" % k["bg"], tile=k["tile"], integrator=kw.get("integrator", "mis"),
            scrambler=kw.get("scrambler", "fastowen"), sampler=kw.get("sampler", "sobol")))
    for key, cfg in CONFIGS:
        wave = cfg.get("waves", [cfg["spp"]])[0]
        out[key] = frame(H.oracle_render(H.scene_file(cfg["scene"], **cfg["kw"]), cfg["w"], cfg["h"], cfg["spp"],
                                         H.scene_camera(cfg["scene"], **cfg["kw"]), first=wave, max=wave,
                                         maxdepth=cfg["max_depth"], tonemap="agx"))
    sp = H.scene_file("soup", **GP.C2["kw"])
    ctx, sel = GP.c2_primary_rays(Y.Scene(sp))
    ctx.close()
    closest = H.oracle_trace(sp, sel, "closest")
    rec = {"rays": H.digest(sel), "closest": GP.hit_digests(closest)}
    sel[:, 7] = np.where(closest["didHit"] == 1, closest["t"] * 0.5, 1e30)
    rec["any"] = H.digest(H.oracle_trace(sp, sel, "any")["didHit"])
    out["c2_soup_hits"] = rec
    for name in ("rgba", "rgb", "grey", "grey_alpha", "smooth_rgb", "palette", "rgb16"):
        png = GL.sample_png(name)
        for t, ch in GL.TEXLOAD_CASES + ((S.NONCOLOR, [0, 1, 2]),):
            out[GL.texload_key(name, t, ch)] = H.digest(H.oracle_texload(png, t, ch))
    for path in ID.LDR[::3]:
        out[f"texload_{os.path.basename(path)}_{S.SRGB}_12"] = H.digest(H.oracle_texload(open(path, "rb").read(), S.SRGB, [1, 2]))
    with tempfile.TemporaryDirectory() as d:
        from pathlib import Path
        glb, _ = GL.build_case(Path(d), check_textures=False)
        ysc, ppm = os.path.join(d, "scene.ysc"), os.path.join(d, "ref.ppm")
        Y.glb_to_ysc(glb, ysc, env=GL.glb_env(), env_radius=80.0)
        ref = H.oracle_render(ysc, 64, 40, 8, GL.GLB_CAM, first=8, max=8, tonemap="agx", ppm=ppm)
        out["glb_scene_64x40_8spp"] = dict(frame(ref), ppm=H.digest(np.fromfile(ppm, np.uint8)))
    return out


def main():
    if not H.have_oracle():
        sys.exit(f"{H.ORACLE} is not built (make -C oracle ref)")
    Y.use_library(H.hostsim())
    Y.default_traversal = Y.TRAVERSAL_REFERENCE_ORDER  # as tests/conftest.py
    out = reference_outputs()
    with open(H.REFERENCE_DIGESTS, "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
        f.write("\n")
    print(f"{len(out)} entries → {H.REFERENCE_DIGESTS}")


if __name__ == "__main__":
    main()
