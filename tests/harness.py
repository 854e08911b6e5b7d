"""Shared test plumbing: the oracle binary (oracle/_ref/oracle_ref = the UNMODIFIED reference),
synthetic scene files, seeded KAT input blobs, the hostsim build, and image metrics.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / reference arm may execute
anything under oracle/.  Nothing here reads /root/reference at run time.
"""
from __future__ import annotations

import hashlib
import json
import os
import struct
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

ORACLE = os.path.join(ROOT, "oracle", "_ref", "oracle_ref")
GOLDEN = os.path.join(ROOT, "tests", "golden")
CACHE = os.environ.get("YART_TEST_CACHE", os.path.join(tempfile.gettempdir(), "yart_b200_test_cache"))
os.makedirs(CACHE, exist_ok=True)


def have_oracle() -> bool:
    return os.path.exists(ORACLE)


def run_oracle(*args, binary=ORACLE, timeout=600) -> str:
    """Runs the oracle binary.  The reference's wave barrier reads `m_currentWave` / `m_waveSamples` outside its
    locks (SURVEY §5) and can deadlock with several threads on tiny frames, hence the timeout + one retry."""
    cmd = [binary, *map(str, args)]
    for attempt in range(2):
        try:
            r = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout)
        except subprocess.TimeoutExpired:
            if attempt == 0:
                continue
            raise RuntimeError(f"oracle_ref {' '.join(map(str, args))} timed out twice")
        if r.returncode != 0:
            raise RuntimeError(f"oracle_ref {' '.join(map(str, args))} failed: {r.stderr}")
        return r.stdout


# ------------------------------------------------------------------------------------------
# scenes
# ------------------------------------------------------------------------------------------
def scene_file(name: str, **kw) -> str:
    """Writes (once) the named synthetic scene as a .ysc file and returns its path."""
    from yart_b200 import scenes
    tag = name + "".join(f"_{k}{v}" for k, v in sorted(kw.items()))
    path = os.path.join(CACHE, tag + ".ysc")
    if not os.path.exists(path):
        s = getattr(scenes, name)(**kw)
        tmp = path + f".tmp{os.getpid()}"
        s.write(tmp)
        os.replace(tmp, path)
    return path


def scene_camera(name: str, **kw) -> dict:
    from yart_b200 import scenes
    if name == "soup":
        kw = dict(kw, n_tris=8)  # camera does not depend on the triangle count
    if name in ("sponza", "mclaren"):
        kw = dict(kw, n_tris=100, env_res=4, **({"tex_res": 4} if name == "sponza" else {}))
    return getattr(scenes, name)(**kw).camera


# ------------------------------------------------------------------------------------------
# oracle commands
# ------------------------------------------------------------------------------------------
def oracle_kat(kind: str, blob: bytes, scene: str | None = None) -> np.ndarray:
    with tempfile.TemporaryDirectory() as d:
        fin, fout = os.path.join(d, "in.bin"), os.path.join(d, "out.bin")
        open(fin, "wb").write(blob)
        args = ["kat", kind, fin, fout] + ([scene] if scene else [])
        run_oracle(*args)
        return np.fromfile(fout, np.float32)


def oracle_trace(scene: str, rays: np.ndarray, mode="closest", usetmax=False) -> np.ndarray:
    from yart_b200 import HIT_DTYPE
    rays = np.ascontiguousarray(rays, np.float32).reshape(-1, 8)
    with tempfile.TemporaryDirectory() as d:
        fin, fout = os.path.join(d, "rays.bin"), os.path.join(d, "hits.bin")
        with open(fin, "wb") as f:
            f.write(struct.pack("<I", len(rays)))
            f.write(rays.tobytes())
        args = ["trace", scene, fin, fout, f"mode={mode}"] + (["usetmax"] if usetmax else [])
        run_oracle(*args)
        return np.fromfile(fout, HIT_DTYPE)


def oracle_render(scene: str, w: int, h: int, spp: int, cam: dict, binary=ORACLE, **kw) -> dict:
    """Returns dict(hdr, ldr (h,w,4), rays, ms, threads, build_ms)."""
    with tempfile.TemporaryDirectory() as d:
        fout = os.path.join(d, "img.bin")
        args = ["render", scene, fout, f"w={w}", f"h={h}", f"spp={spp}",
                "pos=%.17g,%.17g,%.17g" % tuple(cam["pos"]), "target=%.17g,%.17g,%.17g" % tuple(cam["target"]),
                f"focal={cam.get('focal', 35.0)}", f"fnum={cam.get('fnum', 0.0)}", f"exposure={cam.get('exposure', 0.0)}",
                f"sides={cam.get('sides', 0)}"]
        # small frames: one worker thread (the output does not depend on the thread count, and a single thread
        # cannot trip the reference's wave-barrier race); large frames keep the reference's default
        if "threads" not in kw and w * h <= 256 * 256:
            kw = dict(kw, threads=1)
        args += [f"{k}={v}" for k, v in kw.items()]
        run_oracle(*args, binary=binary, timeout=120 if w * h <= 256 * 256 else 900)
        raw = open(fout, "rb").read()
    ww, hh, rays, ms, threads, build_ms = struct.unpack_from("<IIQdId", raw, 0)
    off = struct.calcsize("<IIQdId")
    n = ww * hh * 4
    hdr = np.frombuffer(raw, np.float32, n, off).reshape(hh, ww, 4).copy()
    ldr = np.frombuffer(raw, np.float32, n, off + 4 * n).reshape(hh, ww, 4).copy()
    return dict(hdr=hdr, ldr=ldr, rays=rays, ms=ms, threads=threads, build_ms=build_ms)


def oracle_texload(image: bytes, tex_type: int, channels) -> np.ndarray:
    """The reference's loadTexture<C> on an encoded image: (h, w, C) uint8."""
    with tempfile.TemporaryDirectory() as d:
        fin, fout = os.path.join(d, "image"), os.path.join(d, "out.bin")
        open(fin, "wb").write(image)
        run_oracle("texload", fin, tex_type, len(channels), ",".join(map(str, channels)), fout)
        raw = open(fout, "rb").read()
    w, h, c = struct.unpack_from("<III", raw, 0)
    return np.frombuffer(raw, np.uint8, w * h * c, 12).reshape(h, w, c)


def oracle_bvh(scene: str, kind: str = "sah"):
    with tempfile.TemporaryDirectory() as d:
        fout = os.path.join(d, "bvh.bin")
        run_oracle("bvh", scene, fout, f"kind={kind}")
        raw = open(fout, "rb").read()
    (n_meshes,) = struct.unpack_from("<I", raw, 0)
    off = 4
    dt = np.dtype([("min", "<f4", 3), ("max", "<f4", 3), ("left", "<u4"), ("span", "<u4")])
    out = []
    for _ in range(n_meshes):
        n_nodes, n_tris = struct.unpack_from("<II", raw, off)
        off += 8
        nodes = np.frombuffer(raw, dt, n_nodes, off).copy()
        off += 32 * n_nodes
        idx = np.frombuffer(raw, np.uint32, n_tris, off).copy()
        off += 4 * n_tris
        out.append((nodes, idx))
    return out


# ------------------------------------------------------------------------------------------
# seeded KAT inputs (layouts: oracle/ref_driver.cpp cmdKat)
# ------------------------------------------------------------------------------------------
def _unit(rng, n):
    v = rng.normal(size=(n, 3))
    return (v / np.linalg.norm(v, axis=1, keepdims=True)).astype(np.float32)


def kat_input(kind: str, n: int = 256, seed: int = 7, **kw) -> bytes:
    rng = np.random.default_rng(seed)
    if kind == "sampler":
        spp = kw.get("spp", 16)
        rec = np.stack([rng.integers(0, 4096, n), rng.integers(0, 4096, n), rng.integers(0, spp, n)], 1).astype(np.uint32)
        return struct.pack("<II", spp, n) + rec.tobytes()
    if kind == "lut":
        rec = rng.uniform(0, 1, (n, 4)).astype(np.float32)
        rec[:, 3] = rng.uniform(1.05, 2.5, n)
        rec[::7, 3] = 1.0 / rec[::7, 3]
        rec[::5, 2] = -rec[::5, 2]  # negative cosines: the size_t(negative) behaviour (SURVEY a25)
        rec[::11, 0] = -rec[::11, 0]
        return struct.pack("<I", n) + rec.tobytes()
    if kind == "ggx":
        r = rng.uniform(0.01, 1, (n, 1)).astype(np.float32)
        an = rng.uniform(0, 1, (n, 1)).astype(np.float32)
        an[::2] = 0
        w, wm = _unit(rng, n), _unit(rng, n)
        w[:, 2], wm[:, 2] = np.abs(w[:, 2]) + 1e-3, np.abs(wm[:, 2]) + 1e-3
        u = rng.uniform(0, 1, (n, 2)).astype(np.float32)
        return struct.pack("<I", n) + np.concatenate([r, an, w, wm, u], 1).astype(np.float32).tobytes()
    if kind == "bsdf":
        n_mat = kw["n_materials"]
        nn = _unit(rng, n)
        t = _unit(rng, n)
        t[::9] = 0  # Frame(n) fallback
        wo, wi = _unit(rng, n), _unit(rng, n)
        # mostly upper hemisphere w.r.t. n, some below (transmission / back side)
        flip = (np.einsum("ij,ij->i", wo, nn) < 0) & (rng.uniform(size=n) < 0.8)
        wo[flip] = -wo[flip]
        flip = (np.einsum("ij,ij->i", wi, nn) < 0) & (rng.uniform(size=n) < 0.6)
        wi[flip] = -wi[flip]
        out = bytearray(struct.pack("<I", n))
        for i in range(n):
            out += struct.pack("<I", int(rng.integers(0, n_mat)))
            out += wo[i].tobytes() + wi[i].tobytes() + nn[i].tobytes() + t[i].tobytes()
            out += rng.uniform(-1.5, 2.5, 2).astype(np.float32).tobytes()  # uv (wraps)
            out += rng.uniform(0, 1, 2).astype(np.float32).tobytes()  # u
            out += rng.uniform(0, 1, 2).astype(np.float32).tobytes()  # uc uc2
            out += struct.pack("<I", int(rng.integers(0, 2)))
            out += struct.pack("<ff", 1.0 if rng.uniform() < 0.5 else -1.0, float(rng.uniform(0, 5)))
        return bytes(out)
    if kind in ("light", "lightuniform"):
        n_lights = kw["n_lights"]
        out = bytearray(struct.pack("<I", n))
        p = rng.uniform(-4, 4, (n, 3)).astype(np.float32)
        nn, wi = _unit(rng, n), _unit(rng, n)
        for i in range(n):
            out += struct.pack("<I", int(rng.integers(0, n_lights)))
            out += p[i].tobytes() + nn[i].tobytes() + rng.uniform(0, 1, 2).astype(np.float32).tobytes()
            out += wi[i].tobytes() + struct.pack("<f", float(rng.uniform(0, 1)))
        return bytes(out)
    if kind in ("gmon", "gmonb"):
        ns = kw.get("samples", 16)
        s = rng.gamma(0.5, 2.0, (n, ns, 3)).astype(np.float32)
        s[rng.uniform(size=(n, ns)) < 0.02] *= 500.0  # fireflies
        s[rng.uniform(size=(n, ns)) < 0.01, 0] = np.nan
        s[rng.uniform(size=(n, ns)) < 0.01, 1] = -1.0
        s[: n // 8] = 0.0  # black pixels (G = NaN path)
        return struct.pack("<II", ns, n) + s.tobytes()
    if kind == "agx":
        v = (rng.gamma(0.7, 1.5, (n, 3)) * rng.choice([0.01, 1, 30], (n, 1))).astype(np.float32)
        v[:4] = 0.0
        return struct.pack("<II", kw.get("look", 0), n) + v.tobytes()
    if kind == "camera":
        w, h = kw.get("w", 640), kw.get("h", 360)
        hdr = struct.pack("<IIffI", w, h, kw.get("focal", 35.0), kw.get("fnum", 2.8), kw.get("sides", 0))
        hdr += np.asarray(kw.get("pos", (1, 2, 9)), np.float32).tobytes()
        hdr += np.asarray(kw.get("target", (0, 1, 0)), np.float32).tobytes()
        hdr += np.asarray(kw.get("up", (0, 0, 0)), np.float32).tobytes()
        hdr += struct.pack("<I", n)
        out = bytearray(hdr)
        for i in range(n):
            out += struct.pack("<II", int(rng.integers(0, w)), int(rng.integers(0, h)))
            out += rng.uniform(1e-6, 1, 4).astype(np.float32).tobytes()
        return bytes(out)
    if kind == "texture":
        n_tex = kw["n_textures"]
        out = bytearray(struct.pack("<I", n))
        for i in range(n):
            out += struct.pack("<I", int(rng.integers(0, n_tex)))
            out += rng.uniform(-2, 3, 2).astype(np.float32).tobytes()
        return bytes(out)
    raise KeyError(kind)


KAT_OUT_WORDS = dict(sampler=8, lut=8, ggx=8, bsdf=27, light=22, gmon=9, gmonb=3, lightuniform=3, agx=3, camera=6, texture=4)


def kat_count(kind: str, blob: bytes) -> int:
    if kind in ("sampler", "gmon", "gmonb", "agx"):
        return struct.unpack_from("<I", blob, 4)[0]
    if kind == "camera":
        return struct.unpack_from("<I", blob, 56)[0]
    return struct.unpack_from("<I", blob, 0)[0]


# ------------------------------------------------------------------------------------------
# hostsim (product sources compiled for the CPU — test infrastructure, see tests/hostsim/Makefile)
# ------------------------------------------------------------------------------------------
_hostsim = None


def hostsim():
    global _hostsim
    if _hostsim is None:
        subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "tests", "hostsim")], check=True, capture_output=True)
        from yart_b200 import capi
        _hostsim = capi.load(os.path.join(ROOT, "tests", "hostsim", "libyart_hostsim.so"))
    return _hostsim


# ------------------------------------------------------------------------------------------
# metrics
# ------------------------------------------------------------------------------------------
def rel_mse(img: np.ndarray, ref: np.ndarray, eps: float = 1e-2) -> float:
    """Mean over pixels of |img - ref|^2 / (ref^2 + eps), RGB."""
    a, b = img[..., :3].astype(np.float64), ref[..., :3].astype(np.float64)
    both_nan = np.isnan(a) & np.isnan(b)  # e.g. AgX "punchy": pow(negative, 1.35) is NaN in the reference too
    if (np.isnan(a) != np.isnan(b)).any():
        return float("inf")
    a, b = np.where(both_nan, 0.0, a), np.where(both_nan, 0.0, b)
    return float(np.mean((a - b) ** 2 / (b * b + eps)))


def bits_equal(a: np.ndarray, b: np.ndarray) -> np.ndarray:
    """Bitwise float equality; any NaN equals any NaN (payloads are not part of the contract)."""
    a, b = np.ascontiguousarray(a, np.float32), np.ascontiguousarray(b, np.float32)
    return (a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))


# ------------------------------------------------------------------------------------------
# the reference's outputs recorded as digests (tests/golden/reference_digests.json, record_digests.py next to it):
# equal digests are the bitwise equality bits_equal() checks, without storing full frames
# ------------------------------------------------------------------------------------------
REFERENCE_DIGESTS = os.path.join(GOLDEN, "reference_digests.json")
_recorded = None


def digest(a) -> str:
    """SHA-256 of an array's shape, dtype and bytes, every float NaN replaced by one NaN (bits_equal's rule)."""
    a = np.ascontiguousarray(a)
    if a.dtype.kind == "f":
        a = np.where(np.isnan(a), a.dtype.type(np.nan), a).astype(a.dtype)
    return hashlib.sha256(f"{a.shape}{a.dtype.str}".encode() + a.tobytes()).hexdigest()


def recorded(key: str):
    """The reference's recorded output for one test input: a digest or a dict of digests and counts."""
    global _recorded
    if _recorded is None:
        with open(REFERENCE_DIGESTS) as f:
            _recorded = json.load(f)
    return _recorded[key]
