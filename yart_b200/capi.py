"""ctypes view of include/yart_cuda.h (the C ABI of libyart_b200.so).

Structures and prototypes only; no arithmetic.  `load(path)` binds a shared library that exports
the ABI.  The package default is the CUDA product library next to this file; it raises if that
library is missing or cannot be loaded — there is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
PRODUCT_LIB = os.path.join(HERE, "libyart_b200.so")
# the same sources built with -DYB_RNG_SAMPLERS: adds the Owen / BinaryPermute scramblers and YC_SAMPLER_NAIVE /
# YC_SAMPLER_STRATIFIED (same C ABI)
SAMPLERS_LIB = os.path.join(HERE, "libyart_b200_samplers.so")

YC_OK, YC_ERR_INVALID, YC_ERR_CUDA, YC_ERR_NO_SCENE, YC_ERR_NO_DEVICE, YC_ERR_STATE, YC_ERR_IO = 0, -1, -2, -3, -4, -5, -6
YC_ERR_UNSUPPORTED = -7
TONEMAP_NONE, TONEMAP_AGX, TONEMAP_AGX_GOLDEN, TONEMAP_AGX_PUNCHY = 0, 1, 2, 3
ESTIMATOR_GMON, ESTIMATOR_MON, ESTIMATOR_MEAN, ESTIMATOR_GMONB = 0, 1, 2, 3
TRACE_CLOSEST, TRACE_ANY, TRACE_COUNT, TRACE_USE_TMAX, TRACE_REFERENCE_ORDER, TRACE_WIDE = 0, 1, 16, 32, 64, 128

f32, u32, i32, u64 = C.c_float, C.c_uint32, C.c_int32, C.c_uint64


class YcCamera(C.Structure):
    _fields_ = [("position", f32 * 3), ("topLeftPixel", f32 * 3), ("pixelDeltaU", f32 * 3), ("pixelDeltaV", f32 * 3),
                ("frameX", f32 * 3), ("frameY", f32 * 3), ("frameZ", f32 * 3), ("apertureRadius", f32),
                ("apertureSides", u32), ("exposure", f32)]


BVH_SAH, BVH_MEDIAN_SPLIT, BVH_SAH_DEVICE, BVH_SAH_HOST = 0, 1, 2, 3
INTEGRATOR_MIS, INTEGRATOR_NAIVE = 0, 1
SCRAMBLER_FAST_OWEN, SCRAMBLER_OWEN, SCRAMBLER_BINARY_PERMUTE = 0, 1, 2
SAMPLER_SOBOL, SAMPLER_NAIVE, SAMPLER_STRATIFIED = 0, 1, 2
LIGHT_SAMPLER_POWER, LIGHT_SAMPLER_UNIFORM = 0, 1
TRAVERSAL_AUTO, TRAVERSAL_REFERENCE_ORDER, TRAVERSAL_WIDE = 0, 1, 2


class YcOptions(C.Structure):
    _fields_ = [("maxDepth", u32), ("maxPathsInFlight", u32), ("traceRefillMin", u32), ("traceInnerMin", u32),
                ("tailThreshold", u32), ("integrator", u32), ("scrambler", u32), ("sharedStackEntries", u32),
                ("sampler", u32), ("lightSampler", u32), ("traversal", u32), ("reserved", u32)]


class YcRect(C.Structure):
    _fields_ = [("x", u32), ("y", u32), ("w", u32), ("h", u32)]


class YcFrameDesc(C.Structure):
    _fields_ = [("width", u32), ("height", u32), ("totalSamples", u32), ("tileSize", u32), ("background", f32 * 3),
                ("tonemap", u32), ("estimator", u32), ("shardIndex", u32), ("shardCount", u32)]


class YcStats(C.Structure):
    _fields_ = [("raysReference", u64), ("raysExtend", u64), ("raysShadow", u64), ("samples", u64),
                ("kernelLaunches", u64), ("gpuMs", C.c_double), ("boxTests", u64), ("triTests", u64),
                ("extendMs", C.c_double), ("extendLaunches", u64), ("shadeMs", C.c_double), ("shadeLaunches", u64),
                ("hitsShaded", u64), ("commMs", C.c_double)]


class YcAdaptive(C.Structure):
    _fields_ = [("threshold", f32), ("minSamples", u32), ("lumaFloor", f32), ("reserved", u32)]


class YcRay(C.Structure):
    _fields_ = [("o", f32 * 3), ("tmin", f32), ("d", f32 * 3), ("tmax", f32)]


class YcHit(C.Structure):
    _fields_ = [("t", f32), ("prim", u32), ("material", i32), ("lightIdx", i32), ("backSide", u32), ("didHit", u32),
                ("p", f32 * 3), ("n", f32 * 3), ("tg", f32 * 3), ("uv", f32 * 2), ("attenuation", f32 * 3)]


class YcMesh(C.Structure):
    _fields_ = [("rootMin", f32 * 3), ("rootMax", f32 * 3), ("rootRef", u32), ("nodeOffset", u32), ("triOffset", u32),
                ("vertOffset", u32), ("primOffset", u32), ("nTris", u32), ("nVerts", u32), ("nInner", u32)]


class YcScene(C.Structure):
    _fields_ = [("nodes", C.c_void_p), ("nNodes", u32), ("meshes", C.POINTER(YcMesh)), ("nMeshes", u32),
                ("bvhNodes", C.c_void_p), ("nBvhNodes", u64), ("bvhTris", C.c_void_p), ("nBvhTris", u64),
                ("positions", C.POINTER(f32)), ("normals", C.POINTER(f32)), ("tangents", C.POINTER(f32)),
                ("uvs", C.POINTER(f32)), ("nVerts", u64),
                ("primIndices", C.POINTER(u32)), ("primMaterial", C.POINTER(u32)), ("primLight", C.POINTER(i32)),
                ("nPrims", u64),
                ("materials", C.c_void_p), ("nMaterials", u32), ("textures", C.c_void_p), ("nTextures", u32),
                ("texelsU8", C.c_void_p), ("nTexelsU8", u64), ("texelsF32", C.c_void_p), ("nTexelsF32", u64),
                ("lights", C.c_void_p), ("nLights", u32), ("envDist", C.c_void_p), ("nEnvDist", u64),
                ("infiniteLights", C.POINTER(u32)), ("nInfinite", u32), ("areaLights", C.POINTER(u32)), ("nArea", u32),
                ("lightPowerCdf", C.POINTER(f32)), ("totalPower", f32), ("lutTables", C.POINTER(f32)),
                ("hasAlpha", i32)]


class YrSettings(C.Structure):
    _fields_ = [("width", u32), ("height", u32), ("samples", u32), ("firstWaveSamples", u32), ("maxWaveSamples", u32),
                ("tileSize", u32), ("maxDepth", u32), ("background", f32 * 3), ("tonemap", u32), ("estimator", u32),
                ("shardIndex", u32), ("shardCount", u32), ("device", i32), ("integrator", u32), ("scrambler", u32), ("sampler", u32),
                ("traversal", u32), ("sharding", u32)]


class YrRenderData(C.Structure):
    _fields_ = [("samplesTaken", u64), ("totalSamples", u64), ("totalRays", u64), ("totalTimeMs", C.c_double)]


class YrWaveData(C.Structure):
    _fields_ = [("wave", u64), ("waveSamples", u64), ("rays", u64), ("timeMs", C.c_double)]


class YsEnvLight(C.Structure):
    _fields_ = [("width", u32), ("height", u32), ("rgb", C.POINTER(f32)), ("sceneRadius", f32), ("hasTransform", i32),
                ("transform", f32 * 16)]


class YrTileData(C.Structure):
    _fields_ = [("x", u32), ("y", u32), ("w", u32), ("h", u32), ("index", u64), ("total", u64), ("rays", u64),
                ("timeMs", C.c_double)]


WAVE_CALLBACK = C.CFUNCTYPE(None, C.POINTER(YrRenderData), C.POINTER(YrWaveData), C.c_void_p)
TILE_CALLBACK = C.CFUNCTYPE(None, C.POINTER(YrRenderData), C.POINTER(YrTileData), C.c_void_p)
DONE_CALLBACK = C.CFUNCTYPE(None, C.POINTER(YrRenderData), C.c_int, C.c_void_p)
# yc_collective_fn: fn(buf, count, dtype (0 f32, 1 i32, 2 u64), root (< 0: all), user) → 0 on success
COLLECTIVE_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_void_p)
COMM_ID_BYTES = 128
SHARD_TILES, SHARD_BUCKETS = 0, 1
ERR_ABORTED = -8

P = C.c_void_p
# name → (restype, argtypes): every entry point include/yart_cuda.h declares
PROTOTYPES = {
    "yc_create": (C.c_int, [C.c_int, C.POINTER(YcOptions), C.POINTER(P)]),
    "yc_destroy": (None, [P]),
    "yc_last_error": (C.c_char_p, [P]),
    "yc_upload_scene": (C.c_int, [P, C.POINTER(YcScene)]),
    "yc_set_camera": (C.c_int, [P, C.POINTER(YcCamera)]),
    "yc_set_cameras": (C.c_int, [P, C.POINTER(YcCamera), u32]),
    "yc_begin_frame": (C.c_int, [P, C.POINTER(YcFrameDesc)]),
    "yc_render_wave": (C.c_int, [P, YcRect, u32, u32, u32]),
    "yc_render_wave_async": (C.c_int, [P, YcRect, u32, u32, u32]),
    "yc_wave_sync": (C.c_int, [P]),
    "yc_accumulate_wave": (C.c_int, [P, YcRect, u32, u32, u32, u32]),
    "yc_bucket_device_ptrs": (C.c_int, [P, C.POINTER(P), C.POINTER(C.c_size_t), C.POINTER(u32), C.POINTER(C.c_size_t)]),
    "yc_finalize_wave": (C.c_int, [P, YcRect, u32, u32]),
    "yc_wave_buckets": (C.c_int, [P, u32, C.POINTER(u32)]),
    "yc_resolve": (C.c_int, [P, P, P, C.POINTER(YcStats)]),
    "yc_frame_device_ptrs": (C.c_int, [P, C.POINTER(P), C.POINTER(P), C.POINTER(C.c_size_t)]),
    "yc_retonemap": (C.c_int, [P]),
    "yc_set_profiling": (C.c_int, [P, C.c_int]),
    "yc_trace": (C.c_int, [P, P, C.c_size_t, C.c_int, P, C.POINTER(YcStats)]),
    "yc_trace_device": (C.c_int, [P, P, C.c_size_t, C.c_int, P, C.c_int, C.POINTER(f32)]),
    "yc_device_alloc": (C.c_int, [P, C.c_size_t, C.POINTER(P)]),
    "yc_device_free": (C.c_int, [P, P]),
    "yc_host_alloc": (C.c_int, [P, C.c_size_t, C.POINTER(P)]),
    "yc_host_free": (C.c_int, [P, P]),
    "yc_memcpy_h2d": (C.c_int, [P, P, P, C.c_size_t]),
    "yc_memcpy_d2h": (C.c_int, [P, P, P, C.c_size_t]),
    "yc_generate_primary_rays": (C.c_int, [P, u32, u32, P]),
    "yc_synchronize": (C.c_int, [P]),
    "yc_set_abort_flag": (C.c_int, [P, C.POINTER(i32)]),
    "yc_comm_unique_id": (C.c_int, [P]),
    "yc_comm_init_rank": (C.c_int, [P, C.c_int, C.c_int, P]),
    "yc_comm_init_all": (C.c_int, [C.POINTER(P), C.c_int]),
    "yc_comm_init_custom": (C.c_int, [P, C.c_int, C.c_int, COLLECTIVE_FN, P]),
    "yc_comm_destroy": (C.c_int, [P]),
    "yc_build_bvh_sah": (C.c_int, [C.c_int, P, C.c_size_t, P, C.c_size_t, P, C.POINTER(u32), P, C.POINTER(u32)]),
    "yc_build_last_error": (C.c_char_p, []),
    "yc_comm_reduce_frames": (C.c_int, [P, C.c_int]),
    "yc_comm_reduce_frames_async": (C.c_int, [P, C.c_int]),
    "yc_comm_frames_direct": (C.c_int, [P, C.POINTER(C.c_int)]),
    "yc_resolve_combined": (C.c_int, [P, P, P]),
    "yc_comm_allreduce_buckets": (C.c_int, [P, u32]),
    "yc_comm_sum_u64": (C.c_int, [P, C.POINTER(u64), u32]),
    "yc_enable_aovs": (C.c_int, [P, C.c_int]),
    "yc_resolve_aovs": (C.c_int, [P, P, P]),
    "yc_comm_reduce_aovs": (C.c_int, [P, C.c_int]),
    "yc_resolve_aovs_combined": (C.c_int, [P, P, P]),
    "yc_set_adaptive": (C.c_int, [P, C.POINTER(YcAdaptive)]),
    "yc_resolve_adaptive": (C.c_int, [P, P, P, C.POINTER(u64)]),
    "yc_comm_reduce_adaptive": (C.c_int, [P, C.c_int]),
    "yc_resolve_adaptive_combined": (C.c_int, [P, P, P]),
    "yc_kat": (C.c_int, [P, C.c_char_p, P, C.c_size_t, P, C.c_size_t]),
    "ys_scene_load": (C.c_int, [C.c_char_p, C.POINTER(P)]),
    "ys_scene_load_bvh": (C.c_int, [C.c_char_p, u32, C.POINTER(P)]),
    "ys_set_build_device": (C.c_int, [C.c_int]),
    "ys_scene_device_builds": (u32, [P]),
    "ys_scene_load_glb": (C.c_int, [C.c_char_p, C.POINTER(YsEnvLight), C.POINTER(P)]),
    "ys_glb_convert": (C.c_int, [C.c_char_p, C.c_char_p, C.POINTER(YsEnvLight)]),
    "ys_decode_texture": (C.c_int, [P, C.c_size_t, u32, u32, C.POINTER(i32), P, C.c_size_t, C.POINTER(u32), C.POINTER(u32)]),
    "ys_load_hdr": (C.c_int, [C.c_char_p, C.POINTER(u32), C.POINTER(u32), P, C.c_size_t]),
    "ys_write_ppm": (C.c_int, [C.c_char_p, P, u32, u32]),
    "ys_write_pfm": (C.c_int, [C.c_char_p, P, u32, u32, u32, u32]),
    "ys_scene_destroy": (None, [P]),
    "ys_last_error": (C.c_char_p, []),
    "ys_scene_flat": (C.POINTER(YcScene), [P]),
    "ys_lut_tables": (C.POINTER(f32), [C.POINTER(C.c_size_t)]),
    "ys_scene_build_ms": (C.c_double, [P]),
    "ys_scene_bvh": (C.c_int, [P, u32, C.POINTER(P), C.POINTER(u32), C.POINTER(C.POINTER(u32)), C.POINTER(u32)]),
    "ys_camera_make": (C.c_int, [u32, u32, f32, f32, f32 * 3, f32 * 3, f32 * 3, f32, u32, C.POINTER(YcCamera)]),
    "yr_create": (C.c_int, [C.POINTER(YrSettings), P, C.POINTER(YcCamera), C.POINTER(P)]),
    "yr_create_flat": (C.c_int, [C.POINTER(YrSettings), C.POINTER(YcScene), C.POINTER(YcCamera), C.POINTER(P)]),
    "yr_create_multi": (C.c_int, [C.POINTER(YrSettings), P, C.POINTER(YcCamera), C.POINTER(C.c_int), u32, C.POINTER(P)]),
    "yr_create_multi_flat": (C.c_int, [C.POINTER(YrSettings), C.POINTER(YcScene), C.POINTER(YcCamera), C.POINTER(C.c_int), u32,
                                       C.POINTER(P)]),
    "yr_create_dist": (C.c_int, [C.POINTER(YrSettings), P, C.POINTER(YcCamera), C.c_int, C.c_int, P, C.POINTER(P)]),
    "yr_create_dist_custom": (C.c_int, [C.POINTER(YrSettings), P, C.POINTER(YcCamera), C.c_int, C.c_int, COLLECTIVE_FN, P,
                                        C.POINTER(P)]),
    "yr_destroy": (None, [P]),
    "yr_set_wave_callback": (C.c_int, [P, WAVE_CALLBACK, P]),
    "yr_set_tile_callback": (C.c_int, [P, TILE_CALLBACK, P]),
    "yr_set_done_callback": (C.c_int, [P, DONE_CALLBACK, P]),
    "yr_set_frame_target": (C.c_int, [P, P]),
    "yr_set_camera": (C.c_int, [P, C.POINTER(YcCamera)]),
    "yr_set_cameras": (C.c_int, [P, C.POINTER(YcCamera), u32]),
    "yr_render": (C.c_int, [P]),
    "yr_abort": (C.c_int, [P]),
    "yr_wait": (C.c_int, [P]),
    "yr_render_sync": (C.c_int, [P, C.POINTER(YrRenderData)]),
    "yr_read": (C.c_int, [P, P, P, C.POINTER(YcStats)]),
    "yr_write_ppm": (C.c_int, [P, C.c_char_p]),
    "yr_enable_aovs": (C.c_int, [P, C.c_int]),
    "yr_read_aovs": (C.c_int, [P, P, P]),
    "yr_set_adaptive": (C.c_int, [P, C.POINTER(YcAdaptive)]),
    "yr_read_adaptive": (C.c_int, [P, P, P]),
    "yr_context": (P, [P]),
    "yr_last_error": (C.c_char_p, [P]),
}


def load(path: str = PRODUCT_LIB) -> C.CDLL:
    if not os.path.exists(path):
        raise RuntimeError(
            f"{path} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(make -C yart_b200).  yart_b200 has no CPU fallback.")
    lib = C.CDLL(path)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export the ABI
        fn.restype = res
        fn.argtypes = args
    return lib
