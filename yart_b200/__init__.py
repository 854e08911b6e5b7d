"""yart_b200 — B200 wavefront path tracer behind yart's Scene / Camera / Renderer API.

Python mirror of the host interface in include/yart_cuda.h (which itself mirrors reference
src/core/renderer.hpp:17-104, src/cpu/tile-renderer.hpp:25-38, src/core/camera.hpp:77-136 and
src/gltf/gltf.cpp:319-358).  All work happens in libyart_b200.so (CUDA, sm_100a); this module only
marshals arguments.  Importing it never touches the GPU; creating a Renderer or Context does, and
raises if there is no usable CUDA device — there is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import capi
from .capi import (LIGHT_SAMPLER_POWER, LIGHT_SAMPLER_UNIFORM, SAMPLER_SOBOL, SAMPLER_NAIVE, SAMPLER_STRATIFIED, BVH_SAH, BVH_MEDIAN_SPLIT, BVH_SAH_DEVICE, BVH_SAH_HOST, SCRAMBLER_FAST_OWEN, SCRAMBLER_OWEN, SCRAMBLER_BINARY_PERMUTE, INTEGRATOR_MIS, INTEGRATOR_NAIVE, ESTIMATOR_GMONB, ESTIMATOR_GMON, ESTIMATOR_MEAN, ESTIMATOR_MON, TONEMAP_AGX, TONEMAP_AGX_GOLDEN, TONEMAP_AGX_PUNCHY,
                   TONEMAP_NONE, TRACE_ANY, TRACE_CLOSEST, TRACE_COUNT, TRACE_USE_TMAX, TRACE_REFERENCE_ORDER, TRACE_WIDE,
                   TRAVERSAL_AUTO, TRAVERSAL_REFERENCE_ORDER, TRAVERSAL_WIDE, SHARD_TILES, SHARD_BUCKETS)

_lib = None


def lib():
    """The product library (loaded on first use)."""
    global _lib
    if _lib is None:
        _lib = capi.load()
    return _lib


def use_library(handle):
    """Tests only: bind another build of the same C ABI (tests/hostsim)."""
    global _lib
    _lib = handle


# YcOptions::traversal used by Context / Renderer when none is passed (the bit-exact parity suites set
# TRAVERSAL_REFERENCE_ORDER here; the library's own default is TRAVERSAL_AUTO).
default_traversal = capi.TRAVERSAL_AUTO


class YartError(RuntimeError):
    pass


def _check(rc, what, detail=b""):
    if rc != 0:
        names = {-1: "INVALID", -2: "CUDA", -3: "NO_SCENE", -4: "NO_DEVICE", -5: "STATE", -6: "IO", -7: "UNSUPPORTED",
                 -8: "ABORTED"}
        msg = detail.decode() if isinstance(detail, bytes) else str(detail)
        raise YartError(f"{what} failed: YC_ERR_{names.get(rc, rc)} {msg}")


_NO_DEVICE = b"(no usable CUDA device: yart_b200 has no CPU fallback)"
# yc_create returns UNSUPPORTED only for a sampler variant that the default library folds away
_SAMPLERS_HINT = b"(this build folds the sampler variants away: load capi.SAMPLERS_LIB for the RNG samplers)"


def _f3(v):
    return (C.c_float * 3)(*[float(x) for x in v])


def _env_struct(env, radius, transform):
    if env is None:
        return None, None
    rgb = np.ascontiguousarray(env, np.float32)
    e = capi.YsEnvLight(rgb.shape[1], rgb.shape[0], rgb.ctypes.data_as(C.POINTER(C.c_float)), radius,
                        0 if transform is None else 1)
    if transform is not None:
        e.transform = (C.c_float * 16)(*np.asarray(transform, np.float32).reshape(-1))
    return e, rgb  # keep rgb alive


def set_build_device(device: int):
    """Device the SAH BVH builds of later scene loads run on (-1: host builds only)."""
    lib().ys_set_build_device(int(device))


def comm_init_all(contexts):
    """yc_comm_init_all: the contexts of ONE process become one communicator (each is then driven by its own thread)."""
    arr = (C.c_void_p * len(contexts))(*[c._h for c in contexts])
    _check(lib().yc_comm_init_all(C.cast(arr, C.POINTER(C.c_void_p)), len(contexts)), "yc_comm_init_all")


def comm_unique_id() -> bytes:
    """ncclGetUniqueId through the library (rank 0 calls it and hands the bytes to the other ranks)."""
    buf = (C.c_char * capi.COMM_ID_BYTES)()
    _check(lib().yc_comm_unique_id(buf), "yc_comm_unique_id")
    return bytes(buf)


def glb_to_ysc(glb_path: str, ysc_path: str, env=None, env_radius=100.0, env_transform=None):
    """ys_glb_convert: the GLB loader's result as a .ysc scene description."""
    e, keep = _env_struct(env, env_radius, env_transform)
    rc = lib().ys_glb_convert(glb_path.encode(), ysc_path.encode(), C.byref(e) if e is not None else None)
    _check(rc, f"ys_glb_convert({glb_path})", lib().ys_last_error() or b"")


def decode_texture(png: bytes, tex_type: int, channels) -> np.ndarray:
    """ys_decode_texture: loadTexture<C> (core/texture.hpp:62-90) on an in-memory PNG → (h, w, C) uint8."""
    ch = (C.c_int32 * len(channels))(*channels)
    w, h = C.c_uint32(), C.c_uint32()
    buf = np.frombuffer(png, np.uint8)
    rc = lib().ys_decode_texture(buf.ctypes.data, len(png), tex_type, len(channels), ch, None, 0, C.byref(w), C.byref(h))
    _check(rc, "ys_decode_texture", lib().ys_last_error() or b"")
    out = np.empty((h.value, w.value, len(channels)), np.uint8)
    rc = lib().ys_decode_texture(buf.ctypes.data, len(png), tex_type, len(channels), ch, out.ctypes.data, out.nbytes,
                                 C.byref(w), C.byref(h))
    _check(rc, "ys_decode_texture", lib().ys_last_error() or b"")
    return out


def load_hdr(path: str) -> np.ndarray:
    """loadTextureHDR (texture.cpp:21-35): a Radiance .hdr file as an (h, w, 3) float32 array."""
    w, h = C.c_uint32(), C.c_uint32()
    _check(lib().ys_load_hdr(path.encode(), C.byref(w), C.byref(h), None, 0), f"ys_load_hdr({path})", lib().ys_last_error() or b"")
    out = np.empty((h.value, w.value, 3), np.float32)
    _check(lib().ys_load_hdr(path.encode(), C.byref(w), C.byref(h), out.ctypes.data, out.size), f"ys_load_hdr({path})",
           lib().ys_last_error() or b"")
    return out


def write_ppm(path: str, rgba: np.ndarray):
    rgba = np.ascontiguousarray(rgba, np.float32)
    _check(lib().ys_write_ppm(path.encode(), rgba.ctypes.data, rgba.shape[1], rgba.shape[0]), "ys_write_ppm")


class Scene:
    """yart::Scene built from a .ysc description or a binary glTF file (stands in for gltf::load)."""

    def __init__(self, path: str, env=None, env_radius=100.0, env_transform=None, bvh_kind: int = capi.BVH_SAH):
        self._h = C.c_void_p()
        if path.lower().endswith((".glb", ".gltf")):
            e, keep = _env_struct(env, env_radius, env_transform)
            rc = lib().ys_scene_load_glb(path.encode(), C.byref(e) if e is not None else None, C.byref(self._h))
            _check(rc, f"ys_scene_load_glb({path})", lib().ys_last_error() or b"")
        else:
            rc = lib().ys_scene_load_bvh(path.encode(), bvh_kind, C.byref(self._h))
            _check(rc, f"ys_scene_load_bvh({path})", lib().ys_last_error() or b"")
        self.flat = lib().ys_scene_flat(self._h).contents
        self.build_ms = lib().ys_scene_build_ms(self._h)
        self.device_builds = lib().ys_scene_device_builds(self._h)  # meshes whose SAH BVH was built on the GPU

    def close(self):
        if self._h:
            lib().ys_scene_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def n_tris(self) -> int:
        return int(self.flat.nPrims)

    def bvh(self, mesh: int = 0):
        """(nodes, indices) in the reference's layout: nodes = structured array of 32-byte records."""
        nodes, n_nodes, idx, n_tris = C.c_void_p(), C.c_uint32(), C.POINTER(C.c_uint32)(), C.c_uint32()
        _check(lib().ys_scene_bvh(self._h, mesh, C.byref(nodes), C.byref(n_nodes), C.byref(idx), C.byref(n_tris)),
               "ys_scene_bvh")
        dt = np.dtype([("min", "<f4", 3), ("max", "<f4", 3), ("left", "<u4"), ("span", "<u4")])
        buf = (C.c_char * (32 * n_nodes.value)).from_address(nodes.value)
        return (np.frombuffer(buf, dt).copy(),
                np.ctypeslib.as_array(idx, (n_tris.value,)).copy())


def make_camera(width, height, focal=35.0, fnum=0.0, pos=(0, 0, 5), target=(0, 0, 0), up=(0, 0, 0), exposure=0.0,
                sides=0) -> capi.YcCamera:
    """Camera({w,h}, focal, fnum) + moveAndLookAt(pos, target, up) (camera.hpp:77-136)."""
    cam = capi.YcCamera()
    _check(lib().ys_camera_make(width, height, focal, fnum, _f3(pos), _f3(target), _f3(up), exposure, sides,
                                C.byref(cam)), "ys_camera_make")
    return cam


class Context:
    """Device layer (yc_*): one CUDA context + stream on one GPU."""

    def __init__(self, device: int = 0, max_depth: int = 30, max_paths: int = 0, refill_min: int = 0, inner_min: int = 0,
                 tail_threshold: int = 0, integrator: int = capi.INTEGRATOR_MIS,
                 scrambler: int = capi.SCRAMBLER_FAST_OWEN, sh_stack_entries: int = 0,
                 sampler: int = capi.SAMPLER_SOBOL, light_sampler: int = capi.LIGHT_SAMPLER_POWER,
                 traversal: int | None = None):
        self._h = C.c_void_p()
        traversal = default_traversal if traversal is None else traversal
        opts = capi.YcOptions(maxDepth=max_depth, maxPathsInFlight=max_paths, integrator=integrator, scrambler=scrambler,
                              sampler=sampler, lightSampler=light_sampler, traversal=traversal)
        opts.traceRefillMin, opts.traceInnerMin = refill_min, inner_min  # traversal scheduling knobs (0 = default)
        opts.tailThreshold = 0xffffffff if tail_threshold < 0 else tail_threshold  # tail kernel hand-over (-1 = never)
        opts.sharedStackEntries = sh_stack_entries  # shared traversal-stack entries in use (0 = default; small = spill-path test)
        rc = lib().yc_create(device, C.byref(opts), C.byref(self._h))
        _check(rc, "yc_create", _SAMPLERS_HINT if rc == capi.YC_ERR_UNSUPPORTED else _NO_DEVICE)
        self.frame = None

    def close(self):
        if self._h:
            lib().yc_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc, what):
        _check(rc, what, lib().yc_last_error(self._h) or b"")

    def upload_scene(self, scene: Scene):
        self._ck(lib().yc_upload_scene(self._h, C.byref(scene.flat)), "yc_upload_scene")

    def set_camera(self, cam: capi.YcCamera):
        self._ck(lib().yc_set_camera(self._h, C.byref(cam)), "yc_set_camera")

    def begin_frame(self, width, height, total_samples, tile_size=64, background=(0, 0, 0), tonemap=TONEMAP_AGX,
                    estimator=ESTIMATOR_GMON, shard_index=0, shard_count=1):
        f = capi.YcFrameDesc(width, height, total_samples, tile_size, _f3(background), tonemap, estimator, shard_index,
                             shard_count)
        self._ck(lib().yc_begin_frame(self._h, C.byref(f)), "yc_begin_frame")
        self.frame = f

    def render_wave(self, sample_offset, wave_samples, taken_before, rect=None):
        r = capi.YcRect(0, 0, self.frame.width, self.frame.height) if rect is None else capi.YcRect(*rect)
        self._ck(lib().yc_render_wave(self._h, r, sample_offset, wave_samples, taken_before), "yc_render_wave")

    def render_wave_async(self, sample_offset, wave_samples, taken_before, rect=None):
        """yc_render_wave_async: the wave stays in flight; wave_sync() (or any other call) waits for it."""
        self._ck(lib().yc_render_wave_async(self._h, self._rect(rect), sample_offset, wave_samples, taken_before), "yc_render_wave_async")

    def wave_sync(self):
        self._ck(lib().yc_wave_sync(self._h), "yc_wave_sync")

    def _rect(self, rect):
        return capi.YcRect(0, 0, self.frame.width, self.frame.height) if rect is None else capi.YcRect(*rect)

    def accumulate_wave(self, sample_offset, wave_samples, bucket_shard=0, bucket_shard_count=1, rect=None):
        """Sample loop of a wave into the estimator buckets; with bucket_shard_count > 1 only the samples of
        the buckets b with b % bucket_shard_count == bucket_shard (yc_accumulate_wave)."""
        self._ck(lib().yc_accumulate_wave(self._h, self._rect(rect), sample_offset, wave_samples, bucket_shard,
                                          bucket_shard_count), "yc_accumulate_wave")

    def finalize_wave(self, wave_samples, taken_before, rect=None):
        self._ck(lib().yc_finalize_wave(self._h, self._rect(rect), wave_samples, taken_before), "yc_finalize_wave")

    def wave_buckets(self, wave_samples) -> int:
        m = C.c_uint32()
        self._ck(lib().yc_wave_buckets(self._h, wave_samples, C.byref(m)), "yc_wave_buckets")
        return m.value

    def bucket_device_ptrs(self):
        """(device pointer, bytes, planes, pixels per plane) of the estimator accumulation buffer."""
        p, n, planes, pix = C.c_void_p(), C.c_size_t(), C.c_uint32(), C.c_size_t()
        self._ck(lib().yc_bucket_device_ptrs(self._h, C.byref(p), C.byref(n), C.byref(planes), C.byref(pix)),
                 "yc_bucket_device_ptrs")
        return p.value, n.value, planes.value, pix.value

    def resolve(self, want_hdr=True, want_ldr=True):
        h, w = self.frame.height, self.frame.width
        hdr = np.empty((h, w, 4), np.float32) if want_hdr else None
        ldr = np.empty((h, w, 4), np.float32) if want_ldr else None
        st = capi.YcStats()
        self._ck(lib().yc_resolve(self._h, hdr.ctypes.data if want_hdr else None, ldr.ctypes.data if want_ldr else None,
                                  C.byref(st)), "yc_resolve")
        return hdr, ldr, st

    def stats(self) -> capi.YcStats:
        st = capi.YcStats()
        self._ck(lib().yc_resolve(self._h, None, None, C.byref(st)), "yc_resolve")
        return st

    def frame_device_ptrs(self):
        hdr, ldr, n = C.c_void_p(), C.c_void_p(), C.c_size_t()
        self._ck(lib().yc_frame_device_ptrs(self._h, C.byref(hdr), C.byref(ldr), C.byref(n)), "yc_frame_device_ptrs")
        return hdr.value, ldr.value, n.value

    def retonemap(self):
        self._ck(lib().yc_retonemap(self._h), "yc_retonemap")

    # ---- collectives (yc_comm_*) ----
    def comm_init_rank(self, rank: int, world: int, comm_id: bytes):
        cid = (C.c_char * capi.COMM_ID_BYTES).from_buffer_copy(bytes(comm_id))
        self._ck(lib().yc_comm_init_rank(self._h, rank, world, cid), "yc_comm_init_rank")

    def comm_reduce_frames(self, root: int = 0):
        self._ck(lib().yc_comm_reduce_frames(self._h, root), "yc_comm_reduce_frames")

    def comm_reduce_frames_async(self, root: int = 0):
        self._ck(lib().yc_comm_reduce_frames_async(self._h, root), "yc_comm_reduce_frames_async")

    def comm_frames_direct(self) -> bool:
        """True when the participants store finished pixels straight into the root's frame (peer memory) and
        comm_reduce_frames is only a barrier; False when the frames are summed into the root."""
        d = C.c_int()
        self._ck(lib().yc_comm_frames_direct(self._h, C.byref(d)), "yc_comm_frames_direct")
        return bool(d.value)

    def comm_allreduce_buckets(self, wave_samples: int):
        self._ck(lib().yc_comm_allreduce_buckets(self._h, wave_samples), "yc_comm_allreduce_buckets")

    def resolve_combined(self, want_hdr=True, want_ldr=True):
        h, w = self.frame.height, self.frame.width
        hdr = np.empty((h, w, 4), np.float32) if want_hdr else None
        ldr = np.empty((h, w, 4), np.float32) if want_ldr else None
        self._ck(lib().yc_resolve_combined(self._h, hdr.ctypes.data if want_hdr else None, ldr.ctypes.data if want_ldr else None),
                 "yc_resolve_combined")
        return hdr, ldr

    def set_profiling(self, on: bool):
        """on: bool, or the bit mask of yc_set_profiling (1 extend timing, 2 counting builds, 4 shade timing)."""
        self._ck(lib().yc_set_profiling(self._h, int(on)), "yc_set_profiling")

    def trace(self, rays: np.ndarray, mode=TRACE_CLOSEST):
        """rays: (n, 8) float32 rows {o[3], tmin, d[3], tmax} → (hits structured array, stats)."""
        rays = np.ascontiguousarray(rays, np.float32).reshape(-1, 8)
        hits = np.zeros(len(rays), HIT_DTYPE)
        st = capi.YcStats()
        self._ck(lib().yc_trace(self._h, rays.ctypes.data, len(rays), mode, hits.ctypes.data, C.byref(st)), "yc_trace")
        return hits, st

    def device_alloc(self, nbytes: int) -> int:
        p = C.c_void_p()
        self._ck(lib().yc_device_alloc(self._h, nbytes, C.byref(p)), "yc_device_alloc")
        return p.value

    def device_free(self, ptr: int):
        self._ck(lib().yc_device_free(self._h, ptr), "yc_device_free")

    def h2d(self, dst: int, src: np.ndarray):
        src = np.ascontiguousarray(src)
        self._ck(lib().yc_memcpy_h2d(self._h, dst, src.ctypes.data, src.nbytes), "yc_memcpy_h2d")

    def d2h(self, dst: np.ndarray, src: int):
        self._ck(lib().yc_memcpy_d2h(self._h, dst.ctypes.data, src, dst.nbytes), "yc_memcpy_d2h")

    def generate_primary_rays(self, sample_offset: int, spp: int, rays_dev: int):
        self._ck(lib().yc_generate_primary_rays(self._h, sample_offset, spp, rays_dev), "yc_generate_primary_rays")

    def trace_device(self, rays_dev: int, n: int, hits_dev: int, mode=TRACE_CLOSEST, repeat=1) -> float:
        ms = C.c_float()
        self._ck(lib().yc_trace_device(self._h, rays_dev, n, mode, hits_dev, repeat, C.byref(ms)), "yc_trace_device")
        return ms.value

    def kat(self, kind: str, blob: bytes, out_words: int) -> np.ndarray:
        out = np.zeros(out_words, np.float32)
        buf = np.frombuffer(blob, np.uint8)
        self._ck(lib().yc_kat(self._h, kind.encode(), buf.ctypes.data, len(blob), out.ctypes.data, out.nbytes),
                 f"yc_kat({kind})")
        return out


HIT_DTYPE = np.dtype([("t", "<f4"), ("prim", "<u4"), ("material", "<i4"), ("lightIdx", "<i4"), ("backSide", "<u4"),
                      ("didHit", "<u4"), ("p", "<f4", 3), ("n", "<f4", 3), ("tg", "<f4", 3), ("uv", "<f4", 2),
                      ("attenuation", "<f4", 3)])
COMPACT_HIT_DTYPE = np.dtype([("t", "<f4"), ("u", "<f4"), ("v", "<f4"), ("prim", "<u4"), ("node", "<i4")])


class Renderer:
    """Mirror of cpu::TileRenderer's public surface (tile-renderer.hpp:27-38) + Renderer
    (renderer.hpp:53-95): knobs as attributes, render()/abort()/wait()/render_sync()."""

    def __init__(self, width, height, camera: capi.YcCamera, scene: Scene | None = None, samples=64,
                 first_wave_samples=None, max_wave_samples=None, tile_size=64, max_depth=30, background=(0, 0, 0),
                 tonemap=TONEMAP_AGX, estimator=ESTIMATOR_GMON, shard_index=0, shard_count=1, device=0,
                 integrator=capi.INTEGRATOR_MIS, scrambler=capi.SCRAMBLER_FAST_OWEN, sampler=capi.SAMPLER_SOBOL,
                 traversal=None, sharding=capi.SHARD_TILES, devices=None, dist=None):
        """devices=[g0, g1, ...]: one renderer over several GPUs of this process (yr_create_multi).
        dist=(rank, world, comm): one process per GPU (yr_create_dist); comm = the 128 bytes of comm_unique_id() from
        rank 0, or a callable collective(buf_ptr, count, dtype, root) → 0 (yr_create_dist_custom)."""
        traversal = default_traversal if traversal is None else traversal
        # TileRenderer defaults: samples 64, firstWaveSamples 64, maxWaveSamples 128, tileSize 64 (:11-14)
        s = capi.YrSettings(width, height, samples, 64 if first_wave_samples is None else first_wave_samples,
                            128 if max_wave_samples is None else max_wave_samples, tile_size, max_depth,
                            _f3(background), tonemap, estimator, shard_index, shard_count, device, integrator, scrambler, sampler,
                            traversal, sharding)
        self.settings = s
        self.scene = scene
        self._h = C.c_void_p()
        self._cb = self._tile_cb = self._done_cb = self._coll = None
        sh = scene._h if scene else None
        if devices is not None:
            arr = (C.c_int * len(devices))(*devices)
            rc, what = lib().yr_create_multi(C.byref(s), sh, C.byref(camera), arr, len(devices), C.byref(self._h)), "yr_create_multi"
        elif dist is not None:
            rank, world, comm = dist
            if callable(comm):
                self._coll = capi.COLLECTIVE_FN(lambda buf, count, dtype, root, _u: int(comm(buf, count, dtype, root) or 0))
                rc = lib().yr_create_dist_custom(C.byref(s), sh, C.byref(camera), rank, world, self._coll, None, C.byref(self._h))
            else:
                cid = (C.c_char * capi.COMM_ID_BYTES).from_buffer_copy(bytes(comm)) if comm is not None else None
                rc = lib().yr_create_dist(C.byref(s), sh, C.byref(camera), rank, world, cid, C.byref(self._h))
            what = "yr_create_dist"
        else:
            rc, what = lib().yr_create(C.byref(s), sh, C.byref(camera), C.byref(self._h)), "yr_create"
        _check(rc, what, _NO_DEVICE if rc == capi.YC_ERR_NO_DEVICE else b"")

    def close(self):
        if self._h:
            for p, _ in getattr(self, "_pinned", {}).values():
                lib().yc_host_free(self.context_handle(), p)
            self._pinned = {}
            lib().yr_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc, what):
        _check(rc, what, lib().yr_last_error(self._h) or b"")

    def on_wave_complete(self, fn):
        """fn(render_data: dict, wave_data: dict) — Renderer::onRenderWaveComplete (renderer.hpp:60-75)."""
        def tramp(rd, wd, _user):
            r, w = rd.contents, wd.contents
            fn(dict(samples_taken=r.samplesTaken, total_samples=r.totalSamples, total_rays=r.totalRays,
                    total_time_ms=r.totalTimeMs),
               dict(wave=w.wave, wave_samples=w.waveSamples, rays=w.rays, time_ms=w.timeMs))
        self._cb = capi.WAVE_CALLBACK(tramp)
        self._ck(lib().yr_set_wave_callback(self._h, self._cb, None), "yr_set_wave_callback")

    def on_tile_complete(self, fn):
        """fn(render_data: dict, tile: dict) — Renderer::onRenderTileComplete."""
        def tramp(rd, td, _user):
            r, t = rd.contents, td.contents
            fn(dict(samples_taken=r.samplesTaken, total_samples=r.totalSamples, total_rays=r.totalRays, total_time_ms=r.totalTimeMs),
               dict(x=t.x, y=t.y, w=t.w, h=t.h, index=t.index, total=t.total, rays=t.rays, time_ms=t.timeMs))
        self._tile_cb = capi.TILE_CALLBACK(tramp)
        self._ck(lib().yr_set_tile_callback(self._h, self._tile_cb, None), "yr_set_tile_callback")

    def on_done(self, fn):
        """fn(render_data: dict, aborted: bool) — Renderer::onRenderComplete / onRenderAborted."""
        def tramp(rd, aborted, _user):
            r = rd.contents
            fn(dict(samples_taken=r.samplesTaken, total_samples=r.totalSamples, total_rays=r.totalRays, total_time_ms=r.totalTimeMs),
               bool(aborted))
        self._done_cb = capi.DONE_CALLBACK(tramp)
        self._ck(lib().yr_set_done_callback(self._h, self._done_cb, None), "yr_set_done_callback")

    def set_camera(self, camera: capi.YcCamera):
        self._ck(lib().yr_set_camera(self._h, C.byref(camera)), "yr_set_camera")

    def set_frame_target(self, ldr: np.ndarray):
        """(height, width, 4) float32, C-contiguous: receives the tonemapped frame after every wave, before the callbacks
        (Renderer::m_buffer; yr_set_frame_target).  None detaches."""
        if ldr is not None:
            assert ldr.dtype == np.float32 and ldr.flags.c_contiguous and ldr.size == self.settings.width * self.settings.height * 4
        self._target = ldr
        self._ck(lib().yr_set_frame_target(self._h, ldr.ctypes.data if ldr is not None else None), "yr_set_frame_target")

    def render(self):
        self._ck(lib().yr_render(self._h), "yr_render")

    def abort(self):
        self._ck(lib().yr_abort(self._h), "yr_abort")

    def wait(self) -> bool:
        """Joins the render; False if it was aborted (YC_ERR_ABORTED)."""
        rc = lib().yr_wait(self._h)
        if rc == capi.ERR_ABORTED:
            return False
        self._ck(rc, "yr_wait")
        return True

    def render_sync(self) -> dict:
        d = capi.YrRenderData()
        self._ck(lib().yr_render_sync(self._h, C.byref(d)), "yr_render_sync")
        return dict(samples_taken=d.samplesTaken, total_samples=d.totalSamples, total_rays=d.totalRays,
                    total_time_ms=d.totalTimeMs)

    def _pinned_frame(self, key):
        """A page-locked (h, w, 4) float32 array owned by this renderer (allocated once)."""
        if not hasattr(self, "_pinned"):
            self._pinned = {}
        if key not in self._pinned:
            h, w = self.settings.height, self.settings.width
            p = C.c_void_p()
            _check(lib().yc_host_alloc(self.context_handle(), h * w * 16, C.byref(p)), "yc_host_alloc")
            buf = (C.c_float * (h * w * 4)).from_address(p.value)
            self._pinned[key] = (p, np.frombuffer(buf, np.float32).reshape(h, w, 4))
        return self._pinned[key][1]

    def read(self, want_hdr=True, want_ldr=True, pinned=False):
        h, w = self.settings.height, self.settings.width
        if pinned:
            hdr = self._pinned_frame("hdr") if want_hdr else None
            ldr = self._pinned_frame("ldr") if want_ldr else None
        else:
            hdr = np.empty((h, w, 4), np.float32) if want_hdr else None
            ldr = np.empty((h, w, 4), np.float32) if want_ldr else None
        st = capi.YcStats()
        self._ck(lib().yr_read(self._h, hdr.ctypes.data if want_hdr else None, ldr.ctypes.data if want_ldr else None,
                               C.byref(st)), "yr_read")
        return hdr, ldr, st

    def write_ppm(self, path: str):
        self._ck(lib().yr_write_ppm(self._h, path.encode()), "yr_write_ppm")

    def context_handle(self):
        return lib().yr_context(self._h)

    def frames_direct(self) -> bool:
        """Several GPUs, tile sharding: True when finished pixels are stored straight into the root GPU's frame (peer
        memory) instead of being reduced there (yc_comm_frames_direct; known after the first wave)."""
        d = C.c_int()
        _check(lib().yc_comm_frames_direct(C.c_void_p(lib().yr_context(self._h)), C.byref(d)), "yc_comm_frames_direct")
        return bool(d.value)
