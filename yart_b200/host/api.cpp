// api.cpp — host layer of libyart_b200.so: the C mirror of yart's Scene loading, Camera and
// Renderer API (ys_* / yr_* in include/yart_cuda.h) on top of the device layer (yc_*).
//
//   ys_scene_load     ↔ gltf::load + Mesh/BVH construction      src/gltf/gltf.cpp:319-358, src/core/mesh.hpp:54-61
//   ys_camera_make    ↔ Camera ctor + moveAndLookAt             src/core/camera.hpp:25-59, 77-136
//   yr_render / yr_render_sync / yr_abort / yr_wait
//                     ↔ Renderer::render / renderSync / abort / wait   src/core/renderer.hpp:56-95
//   wave schedule     ↔ TileRenderer::renderImpl / finishTile   src/cpu/tile-renderer.hpp:118-124, 264-288
// Compiled with g++ -ffp-contract=off (derived constants must round like the reference's).
#include <atomic>
#include <chrono>
#include <cmath>
#include <mutex>
#include <new>
#include <thread>
#include <cstring>
#include <vector>

#include "scene.hpp"

using namespace yartb;

namespace yartb {
bool loadGlb(const std::string& path, ysc::SceneDesc& out, std::string* err);
bool writePpm(const std::string& path, const float* rgba, uint32_t w, uint32_t h);
bool decodeTextureForTest(const uint8_t* png, size_t len, uint32_t type, int C, const int* channels, ysc::TextureDesc& out,
                          std::string& err);
bool decodeRadianceHdr(const uint8_t* data, size_t len, int& w, int& h, std::vector<float>& rgb, std::string& err);
}  // namespace yartb

struct ys_scene {
  HostScene host;
};

static thread_local std::string g_ysError;

// Nothing may throw across the C ABI: allocation failures and container errors raised while loading a (possibly
// hostile) file become error codes.
template <class F>
static int guarded(F&& body) {
  try {
    return body();
  } catch (const std::bad_alloc&) {
    g_ysError = "out of memory";
    return YC_ERR_IO;
  } catch (const std::exception& e) {
    g_ysError = std::string("internal error: ") + e.what();
    return YC_ERR_INVALID;
  } catch (...) {
    g_ysError = "internal error";
    return YC_ERR_INVALID;
  }
}

extern "C" const char* ys_last_error(void) { return g_ysError.c_str(); }

extern "C" int ys_scene_load_bvh(const char* path, uint32_t bvhKind, ys_scene** out);
extern "C" int ys_scene_load(const char* path, ys_scene** out) { return ys_scene_load_bvh(path, YS_BVH_SAH, out); }

extern "C" int ys_scene_load_bvh(const char* path, uint32_t bvhKind, ys_scene** out) {
  return guarded([&]() -> int {
    if (!path || !out || bvhKind > YS_BVH_SAH_HOST) return YC_ERR_INVALID;
    *out = nullptr;
    ysc::SceneDesc d;
    std::string err;
    if (!ysc::load(path, d, &err)) {
      g_ysError = err;
      return YC_ERR_IO;
    }
    ys_scene* s = new (std::nothrow) ys_scene();
    if (!s) return YC_ERR_INVALID;
    s->host.bvhKind = bvhKind;
    if (!s->host.build(d, &err)) {
      g_ysError = err;
      delete s;
      return YC_ERR_INVALID;
    }
    *out = s;
    return YC_OK;
  });
}

// main.cpp:81-84: `ImageInfiniteLight(radius, &hdri); scene->addLight(...)` after gltf::load
static void appendEnv(ysc::SceneDesc& d, const YsEnvLight* env) {
  if (!env || !env->rgb || env->width < 2 || env->height < 2) return;
  ysc::TextureDesc t;
  t.channels = 3, t.isFloat = 1, t.type = ysc::LinearRGB, t.width = env->width, t.height = env->height;
  t.f32.assign(env->rgb, env->rgb + size_t(env->width) * env->height * 3);
  d.textures.push_back(std::move(t));
  ysc::LightDesc l;
  l.type = ysc::ImageInfiniteT;
  l.hdrTex = int32_t(d.textures.size()) - 1;
  l.sceneRadius = env->sceneRadius;
  l.hasTransform = env->hasTransform;
  if (env->hasTransform) memcpy(l.m, env->transform, sizeof l.m);
  d.lights.push_back(l);
}

extern "C" int ys_glb_convert(const char* glbPath, const char* yscPath, const YsEnvLight* env) {
  return guarded([&]() -> int {
    if (!glbPath || !yscPath) return YC_ERR_INVALID;
    ysc::SceneDesc d;
    std::string err;
    if (!loadGlb(glbPath, d, &err)) {
      g_ysError = err;
      return YC_ERR_IO;
    }
    appendEnv(d, env);
    if (!ysc::save(yscPath, d)) {
      g_ysError = std::string("cannot write ") + yscPath;
      return YC_ERR_IO;
    }
    return YC_OK;
  });
}

extern "C" int ys_scene_load_glb(const char* path, const YsEnvLight* env, ys_scene** out) {
  return guarded([&]() -> int {
    if (!path || !out) return YC_ERR_INVALID;
    *out = nullptr;
    ysc::SceneDesc d;
    std::string err;
    if (!loadGlb(path, d, &err)) {
      g_ysError = err;
      return YC_ERR_IO;
    }
    appendEnv(d, env);
    ys_scene* s = new (std::nothrow) ys_scene();
    if (!s) return YC_ERR_INVALID;
    if (!s->host.build(d, &err)) {
      g_ysError = err;
      delete s;
      return YC_ERR_INVALID;
    }
    *out = s;
    return YC_OK;
  });
}

extern "C" int ys_decode_texture(const void* png, size_t len, uint32_t type, uint32_t nChannels, const int32_t* channels,
                                 uint8_t* out, size_t outBytes, uint32_t* width, uint32_t* height) {
  return guarded([&]() -> int {
    if (!png || !channels || nChannels < 1 || nChannels > 4) return YC_ERR_INVALID;
    ysc::TextureDesc t;
    std::string err;
    int ch[4] = {0, 1, 2, 3};
    for (uint32_t i = 0; i < nChannels; i++) ch[i] = channels[i];
    if (!decodeTextureForTest(static_cast<const uint8_t*>(png), len, type, int(nChannels), ch, t, err)) {
      g_ysError = err;
      return YC_ERR_IO;
    }
    if (width) *width = t.width;
    if (height) *height = t.height;
    if (out) {
      if (outBytes < t.u8.size()) return YC_ERR_INVALID;
      memcpy(out, t.u8.data(), t.u8.size());
    }
    return YC_OK;
  });
}

// loadTextureHDR(filename) (src/core/texture.cpp:21-35): the environment map main.cpp:81 hands to ImageInfiniteLight
extern "C" int ys_load_hdr(const char* path, uint32_t* width, uint32_t* height, float* rgb, size_t rgbFloats) {
  if (!path || !width || !height) return YC_ERR_INVALID;
  return guarded([&]() -> int {
    FILE* f = fopen(path, "rb");
    if (!f) {
      g_ysError = std::string("cannot open ") + path;
      return YC_ERR_IO;
    }
    std::vector<uint8_t> buf;
    uint8_t chunk[65536];
    for (size_t n; (n = fread(chunk, 1, sizeof chunk, f)) > 0;) buf.insert(buf.end(), chunk, chunk + n);
    fclose(f);
    int w = 0, h = 0;
    std::vector<float> px;
    std::string err;
    if (!decodeRadianceHdr(buf.data(), buf.size(), w, h, px, err)) {
      g_ysError = err + " in " + path;
      return YC_ERR_IO;
    }
    *width = uint32_t(w), *height = uint32_t(h);
    if (rgb) {
      if (rgbFloats < px.size()) return YC_ERR_INVALID;
      memcpy(rgb, px.data(), px.size() * sizeof(float));
    }
    return YC_OK;
  });
}

extern "C" int ys_write_ppm(const char* path, const float* rgba, uint32_t width, uint32_t height) {
  if (!path || !rgba || !width || !height) return YC_ERR_INVALID;
  return writePpm(path, rgba, width, height) ? YC_OK : YC_ERR_IO;
}

// Portable Float Map: "PF" (RGB) or "Pf" (grey) header, negative scale = little-endian, rows from the bottom up.
extern "C" int ys_write_pfm(const char* path, const float* data, uint32_t width, uint32_t height, uint32_t strideFloats,
                            uint32_t channels) {
  if (!path || !data || !width || !height || (channels != 1 && channels != 3) || strideFloats < channels) return YC_ERR_INVALID;
  return guarded([&]() -> int {
    FILE* f = fopen(path, "wb");
    if (!f) {
      g_ysError = std::string("cannot write ") + path;
      return YC_ERR_IO;
    }
    bool ok = fprintf(f, "%s\n%u %u\n-1.0\n", channels == 3 ? "PF" : "Pf", width, height) > 0;
    std::vector<uint8_t> row(size_t(width) * channels * 4);
    for (uint32_t y = height; ok && y-- > 0;) {
      uint8_t* o = row.data();
      for (uint32_t x = 0; x < width; x++)
        for (uint32_t c = 0; c < channels; c++) {
          uint32_t u;
          memcpy(&u, data + (size_t(y) * width + x) * strideFloats + c, 4);
          for (int k = 0; k < 4; k++) *o++ = uint8_t(u >> (8 * k));
        }
      ok = fwrite(row.data(), 1, row.size(), f) == row.size();
    }
    ok = (fclose(f) == 0) && ok;
    if (!ok) g_ysError = std::string("cannot write ") + path;
    return ok ? YC_OK : YC_ERR_IO;
  });
}

extern "C" void ys_scene_destroy(ys_scene* s) { delete s; }
extern "C" const YcScene* ys_scene_flat(const ys_scene* s) { return s ? &s->host.flat : nullptr; }
extern "C" double ys_scene_build_ms(const ys_scene* s) { return s ? s->host.buildMs : 0.0; }
extern "C" uint32_t ys_scene_device_builds(const ys_scene* s) { return s ? s->host.deviceBuilds : 0u; }
extern "C" int ys_set_build_device(int device) { return yartb::setBuildDevice(device); }

extern "C" int ys_scene_bvh(const ys_scene* s, uint32_t mesh, const void** nodes, uint32_t* nNodes,
                            const uint32_t** indices, uint32_t* nTris) {
  if (!s || mesh >= s->host.refBvh.size()) return YC_ERR_INVALID;
  const BvhBuildResult& b = s->host.refBvh[mesh];
  if (nodes) *nodes = b.nodes.data();
  if (nNodes) *nNodes = uint32_t(b.nodes.size());
  if (indices) *indices = b.indices.data();
  if (nTris) *nTris = uint32_t(b.indices.size());
  return YC_OK;
}

// Camera(imageSize, focalLength, fNumber) with the default 36x24 sensor, then moveAndLookAt
// (camera.hpp:131-136 → setDirection :98-105 → calcDerivedProperties :25-59).
extern "C" int ys_camera_make(uint32_t width, uint32_t height, float focalLength, float fNumber, const float position[3],
                              const float target[3], const float up[3], float exposure, uint32_t apertureSides,
                              YcCamera* out) {
  if (!out || !position || !target || width == 0 || height == 0) return YC_ERR_INVALID;
  const float sensorX = 36.0f, sensorY = 24.0f;
  const f3 pos(position), forward = f3(target) - f3(position);
  f3 mUp(0.0f, 1.0f, 0.0f);
  if (up && length2(f3(up)) != 0.0f) mUp = f3(up);
  const float aspect = float(width) / float(height);
  const float sensorAspect = sensorX / sensorY;
  const float croppedSensorHeight = sensorX / rmax(sensorAspect, aspect);
  const float focusDistance = length(forward);
  const float vh = focusDistance * croppedSensorHeight / focalLength;
  const float vw = vh * aspect;
  mUp = normalized(mUp);
  const f3 w = normalized(-forward);
  const f3 u = cross(mUp, w);
  const f3 v = cross(w, u);
  const Frame frame(w, u);
  const f3 viewportU = u * vw;
  const f3 viewportV = (-v) * vh;
  const f3 viewportTopLeft = pos - w * focusDistance - (viewportU + viewportV) * 0.5f;
  const f3 pixelDeltaU = viewportU / float(width);
  const f3 pixelDeltaV = viewportV / float(height);
  const f3 topLeftPixel = viewportTopLeft + (pixelDeltaU + pixelDeltaV) * 0.5f;
  const float apertureRadius = fNumber ? (focalLength / 2000.0f) / fNumber : 0.0f;
  auto put = [](float* d, f3 s) { d[0] = s.x, d[1] = s.y, d[2] = s.z; };
  put(out->position, pos);
  put(out->topLeftPixel, topLeftPixel);
  put(out->pixelDeltaU, pixelDeltaU);
  put(out->pixelDeltaV, pixelDeltaV);
  put(out->frameX, frame.x);
  put(out->frameY, frame.y);
  put(out->frameZ, frame.z);
  out->apertureRadius = apertureRadius;
  out->apertureSides = apertureSides;
  out->exposure = exposure;
  return YC_OK;
}

// ---------------------------------------------------------------------------------------
// renderer
// ---------------------------------------------------------------------------------------
// One shard per GPU this process drives: a device context and whether the scene is resident there.
struct Shard {
  yc_ctx* ctx = nullptr;
  int device = 0;
  bool sceneUploaded = false;
};

struct yr_renderer {
  YrSettings s{};
  const YcScene* flat = nullptr;  // the scene (owned by a ys_scene or by the caller of yr_create_flat)
  std::vector<YcCamera> cams;     // one per view (yr_set_cameras)
  uint32_t frameViews = 1;        // the view count of the current (or last) render's frame
  std::vector<Shard> shards;      // 1, or one per GPU of yr_create_multi
  // sharding across `world` participants: the local shards are ranks rank0 .. rank0 + shards.size() - 1
  uint32_t rank0 = 0, world = 1;
  bool comm = false;              // yc_comm_* is initialised on every shard (world > 1)
  std::string err;
  yr_wave_callback cb = nullptr;
  void* cbUser = nullptr;
  yr_tile_callback tileCb = nullptr;
  void* tileUser = nullptr;
  yr_done_callback doneCb = nullptr;
  void* doneUser = nullptr;
  float* target = nullptr;        // host frame every wave is copied into before the callbacks (Renderer::m_buffer)
  std::thread worker;
  int32_t stop = 0;               // polled by the device layer between chunks and bounces (yc_set_abort_flag)
  std::mutex m;
  YrRenderData last{};
  int lastRc = YC_OK;
  bool aovs = false;                // yr_enable_aovs
  bool adaptive = false;            // yr_set_adaptive
  YcAdaptive adParams{};
  std::atomic<bool> running{false}; // a render is in progress (yr_render's worker, or yr_render_sync)
};

static int rfail(yr_renderer* r, int rc, const std::string& msg) {
  r->err = msg;
  return rc;
}

static int createShards(yr_renderer* r, const int* devices, uint32_t n) {
  YcOptions o{};
  o.maxDepth = r->s.maxDepth;
  o.integrator = r->s.integrator;
  o.scrambler = r->s.scrambler;
  o.sampler = r->s.sampler;
  o.traversal = r->s.traversal;
  r->shards.resize(n);
  for (uint32_t i = 0; i < n; i++) {
    r->shards[i].device = devices[i];
    const int rc = yc_create(devices[i], &o, &r->shards[i].ctx);
    if (rc != YC_OK) return rc;
    yc_set_abort_flag(r->shards[i].ctx, &r->stop);
  }
  return YC_OK;
}

static void destroyRenderer(yr_renderer* r) {
  for (Shard& sh : r->shards)
    if (sh.ctx) yc_destroy(sh.ctx);  // releases its communicator too
  delete r;
}

static int newRenderer(const YrSettings* settings, const YcScene* flat, const YcCamera* camera, yr_renderer** out) {
  if (!settings || !camera || !out) return YC_ERR_INVALID;
  *out = nullptr;
  if (settings->width == 0 || settings->height == 0 || settings->samples == 0 || settings->tileSize == 0 ||
      settings->sharding > YR_SHARD_BUCKETS)
    return YC_ERR_INVALID;
  yr_renderer* r = new (std::nothrow) yr_renderer();
  if (!r) return YC_ERR_INVALID;
  r->s = *settings;
  r->flat = flat;
  r->cams.assign(camera, camera + 1);
  *out = r;
  return YC_OK;
}

extern "C" int yr_create_flat(const YrSettings* settings, const YcScene* scene, const YcCamera* camera, yr_renderer** out) {
  yr_renderer* r = nullptr;
  int rc = newRenderer(settings, scene, camera, &r);
  if (rc != YC_OK) return rc;
  // YrSettings::shardIndex / shardCount: the caller combines the shards' frames itself (tile sharding, frames sum)
  r->rank0 = settings->shardIndex, r->world = settings->shardCount ? settings->shardCount : 1;
  if ((rc = createShards(r, &settings->device, 1)) != YC_OK) {
    destroyRenderer(r);
    return rc;
  }
  *out = r;
  return YC_OK;
}

extern "C" int yr_create(const YrSettings* settings, const ys_scene* scene, const YcCamera* camera, yr_renderer** out) {
  return yr_create_flat(settings, scene ? ys_scene_flat(scene) : nullptr, camera, out);
}

extern "C" int yr_create_multi_flat(const YrSettings* settings, const YcScene* scene, const YcCamera* camera, const int* devices,
                                    uint32_t nDevices, yr_renderer** out) {
  if (!devices || nDevices == 0 || nDevices > 64) return YC_ERR_INVALID;
  yr_renderer* r = nullptr;
  int rc = newRenderer(settings, scene, camera, &r);
  if (rc != YC_OK) return rc;
  r->rank0 = 0, r->world = nDevices;
  if ((rc = createShards(r, devices, nDevices)) != YC_OK) {
    destroyRenderer(r);
    return rc;
  }
  if (nDevices > 1) {
    std::vector<yc_ctx*> ctxs;
    for (Shard& sh : r->shards) ctxs.push_back(sh.ctx);
    if ((rc = yc_comm_init_all(ctxs.data(), int(nDevices))) != YC_OK) {
      destroyRenderer(r);
      return rc;
    }
    r->comm = true;
  }
  *out = r;
  return YC_OK;
}

extern "C" int yr_create_multi(const YrSettings* settings, const ys_scene* scene, const YcCamera* camera, const int* devices,
                               uint32_t nDevices, yr_renderer** out) {
  return yr_create_multi_flat(settings, scene ? ys_scene_flat(scene) : nullptr, camera, devices, nDevices, out);
}

static int createDist(const YrSettings* settings, const ys_scene* scene, const YcCamera* camera, int rank, int world,
                      const void* commId, yc_collective_fn fn, void* user, yr_renderer** out) {
  if (rank < 0 || world < 1 || rank >= world || (world > 1 && !commId && !fn)) return YC_ERR_INVALID;
  yr_renderer* r = nullptr;
  int rc = newRenderer(settings, scene ? ys_scene_flat(scene) : nullptr, camera, &r);
  if (rc != YC_OK) return rc;
  r->rank0 = uint32_t(rank), r->world = uint32_t(world);
  if ((rc = createShards(r, &settings->device, 1)) != YC_OK) {
    destroyRenderer(r);
    return rc;
  }
  if (world > 1) {
    rc = fn ? yc_comm_init_custom(r->shards[0].ctx, rank, world, fn, user) : yc_comm_init_rank(r->shards[0].ctx, rank, world, commId);
    if (rc != YC_OK) {
      destroyRenderer(r);
      return rc;
    }
    r->comm = true;
  }
  *out = r;
  return YC_OK;
}

extern "C" int yr_create_dist(const YrSettings* settings, const ys_scene* scene, const YcCamera* camera, int rank, int world,
                              const void* commId, yr_renderer** out) {
  return createDist(settings, scene, camera, rank, world, commId, nullptr, nullptr, out);
}

extern "C" int yr_create_dist_custom(const YrSettings* settings, const ys_scene* scene, const YcCamera* camera, int rank, int world,
                                     yc_collective_fn fn, void* user, yr_renderer** out) {
  if (!fn) return YC_ERR_INVALID;
  return createDist(settings, scene, camera, rank, world, nullptr, fn, user, out);
}

extern "C" void yr_destroy(yr_renderer* r) {
  if (!r) return;
  r->stop = 1;
  if (r->worker.joinable()) r->worker.join();
  destroyRenderer(r);
}

extern "C" int yr_set_wave_callback(yr_renderer* r, yr_wave_callback cb, void* user) {
  if (!r) return YC_ERR_INVALID;
  r->cb = cb;
  r->cbUser = user;
  return YC_OK;
}
extern "C" int yr_set_tile_callback(yr_renderer* r, yr_tile_callback cb, void* user) {
  if (!r) return YC_ERR_INVALID;
  r->tileCb = cb;
  r->tileUser = user;
  return YC_OK;
}
extern "C" int yr_set_done_callback(yr_renderer* r, yr_done_callback cb, void* user) {
  if (!r) return YC_ERR_INVALID;
  r->doneCb = cb;
  r->doneUser = user;
  return YC_OK;
}
extern "C" int yr_set_frame_target(yr_renderer* r, float* ldrRGBA) {
  if (!r) return YC_ERR_INVALID;
  r->target = ldrRGBA;
  return YC_OK;
}
extern "C" int yr_set_cameras(yr_renderer* r, const YcCamera* cams, uint32_t n) {
  if (!r || !cams || n == 0 || n > 65535) return YC_ERR_INVALID;
  if (r->worker.joinable()) r->worker.join();
  r->cams.assign(cams, cams + n);
  return YC_OK;
}

extern "C" int yr_set_camera(yr_renderer* r, const YcCamera* cam) { return yr_set_cameras(r, cam, 1); }

// Rows of the current (or last) render's frame: its views stacked.
static uint32_t frameRows(const yr_renderer* r) { return r->s.height * r->frameViews; }

extern "C" yc_ctx* yr_context(yr_renderer* r) { return r && !r->shards.empty() ? r->shards[0].ctx : nullptr; }
extern "C" const char* yr_last_error(const yr_renderer* r) { return r ? r->err.c_str() : "null renderer"; }

// Runs fn(shard index) on every local shard — inline for one, one driver thread per GPU otherwise — and returns the
// first failure (YC_ERR_ABORTED only if nothing worse happened).
template <class F>
static int onShards(yr_renderer* r, F fn) {
  const size_t n = r->shards.size();
  std::vector<int> rc(n, YC_OK);
  if (n == 1) {
    rc[0] = fn(0);
  } else {
    std::vector<std::thread> th;
    for (size_t i = 0; i < n; i++) th.emplace_back([&, i] { rc[i] = fn(i); });
    for (auto& t : th) t.join();
  }
  int out = YC_OK;
  for (size_t i = 0; i < n; i++)
    if (rc[i] != YC_OK && (out == YC_OK || out == YC_ERR_ABORTED)) {
      out = rc[i];
      if (rc[i] != YC_ERR_ABORTED) r->err = yc_last_error(r->shards[i].ctx);
    }
  return out;
}

static bool rootHere(const yr_renderer* r) { return r->rank0 == 0; }

// The frame as the caller sees it: one context's own frames, or the combination of all shards' on the root.
static int readFrames(yr_renderer* r, float* hdr, float* ldr) {
  yc_ctx* c0 = r->shards[0].ctx;
  if (r->comm && r->s.sharding == YR_SHARD_TILES) return rootHere(r) ? yc_resolve_combined(c0, hdr, ldr) : YC_OK;
  return yc_resolve(c0, hdr, ldr, nullptr);
}

static int renderBlocking(yr_renderer* r, YrRenderData* out) {
  using clock = std::chrono::high_resolution_clock;
  if (!r->flat) return rfail(r, YC_ERR_NO_SCENE, "no scene (reference: `if (!scene) return;`, integrator.cpp:6)");
  const bool buckets = r->comm && r->s.sharding == YR_SHARD_BUCKETS;
  r->frameViews = uint32_t(r->cams.size());
  int rc = onShards(r, [&](size_t i) {
    Shard& sh = r->shards[i];
    int e;
    if (!sh.sceneUploaded) {
      if ((e = yc_upload_scene(sh.ctx, r->flat)) != YC_OK) return e;
      sh.sceneUploaded = true;
    }
    if ((e = yc_set_cameras(sh.ctx, r->cams.data(), uint32_t(r->cams.size()))) != YC_OK) return e;
    YcFrameDesc f{};
    f.width = r->s.width, f.height = r->s.height;
    f.totalSamples = r->s.samples, f.tileSize = r->s.tileSize;
    for (int k = 0; k < 3; k++) f.background[k] = r->s.background[k];
    f.tonemap = r->s.tonemap, f.estimator = r->s.estimator;
    // tile sharding: this shard renders the tiles with index % world == its rank; bucket sharding: every shard holds
    // the whole frame and takes its (bucket, pixel class) units of every wave
    f.shardIndex = buckets ? 0u : r->rank0 + uint32_t(i), f.shardCount = buckets ? 1u : r->world;
    if ((e = yc_begin_frame(sh.ctx, &f)) != YC_OK) return e;
    if ((e = yc_set_adaptive(sh.ctx, r->adaptive ? &r->adParams : nullptr)) != YC_OK) return e;
    return yc_enable_aovs(sh.ctx, r->aovs ? 1 : 0);
  });
  if (rc != YC_OK) return rfail(r, rc, r->err);

  // wave schedule: tile-renderer.hpp:120-124 (reset) and :264-288 (advance)
  const uint64_t total = r->s.samples;
  uint64_t remaining = total, wave = 0;
  uint64_t waveSamples = std::min<uint64_t>(r->s.firstWaveSamples ? r->s.firstWaveSamples : total, total);
  const uint64_t maxWave = r->s.maxWaveSamples ? r->s.maxWaveSamples : total;
  const auto t0 = clock::now();
  YrRenderData data{};
  data.totalSamples = total;
  uint64_t raysBefore = 0;
  bool aborted = false;
  const YcRect full{0, 0, r->s.width, frameRows(r)};
  while (waveSamples > 0) {
    const auto w0 = clock::now();
    const uint32_t taken = uint32_t(total - remaining), ws = uint32_t(waveSamples);
    // the sample loop of the wave on every shard, concurrently
    rc = onShards(r, [&](size_t i) {
      yc_ctx* c = r->shards[i].ctx;
      return buckets ? yc_accumulate_wave(c, full, taken, ws, r->rank0 + uint32_t(i), r->world) : yc_render_wave(c, full, taken, ws, taken);
    });
    if (rc != YC_OK && rc != YC_ERR_ABORTED) return rfail(r, rc, r->err);
    // rays of the wave over all participants, whether anyone was told to stop, and the pixels still sampling (adaptive
    // sampling): agreed on collectively, so that either every participant enters the wave's data collective or none does
    uint64_t agree[3] = {0, uint64_t(rc == YC_ERR_ABORTED || r->stop != 0), 0};
    for (Shard& sh : r->shards) {
      YcStats st{};
      yc_resolve(sh.ctx, nullptr, nullptr, &st);
      agree[0] += st.raysReference;
      uint64_t active = 0;
      if (r->adaptive && !agree[1] && (rc = yc_resolve_adaptive(sh.ctx, nullptr, nullptr, &active)) != YC_OK)
        return rfail(r, rc, yc_last_error(sh.ctx));
      agree[2] += active;
    }
    if (r->comm && r->shards.size() == 1) {  // one process per GPU: sum over the ranks
      if ((rc = yc_comm_sum_u64(r->shards[0].ctx, agree, 3)) != YC_OK) return rfail(r, rc, yc_last_error(r->shards[0].ctx));
    }
    if (agree[1]) {
      aborted = true;
      break;
    }
    if (r->comm) {
      rc = onShards(r, [&](size_t i) {
        yc_ctx* c = r->shards[i].ctx;
        if (!buckets) return yc_comm_reduce_frames(c, 0);
        const int e = yc_comm_allreduce_buckets(c, ws);
        return e != YC_OK ? e : yc_finalize_wave(c, full, ws, taken);
      });
      if (rc != YC_OK) return rfail(r, rc, r->err);
    }
    remaining -= waveSamples;
    const auto now = clock::now();
    data.samplesTaken = total - remaining;
    data.totalRays = agree[0];  // of this render (TileRenderer::m_totalRays keeps growing over renderSync calls)
    data.totalTimeMs = std::chrono::duration<double, std::milli>(now - t0).count();
    if (r->target && (!r->comm || rootHere(r)))
      if ((rc = readFrames(r, nullptr, r->target)) != YC_OK) return rfail(r, rc, yc_last_error(r->shards[0].ctx));
    const uint64_t waveRays = agree[0] - raysBefore;
    const double waveMs = std::chrono::duration<double, std::milli>(now - w0).count();
    if (r->tileCb) {
      // the reference reports every tile of every wave (finishTile, tile-renderer.hpp:205-262); a wave here covers the
      // frame at once, so the tiles are reported after it, in tile-list order (view after view, in stacked
      // coordinates), with the wave's rays and time shared out by pixel count
      const uint32_t ts = r->s.tileSize, tilesX = (r->s.width + ts - 1) / ts, tilesY = (r->s.height + ts - 1) / ts;
      const uint32_t views = r->frameViews;
      const double px = double(r->s.width) * frameRows(r);
      for (uint32_t v = 0; v < views; v++)
        for (uint32_t ty = 0; ty < tilesY; ty++)
          for (uint32_t tx = 0; tx < tilesX; tx++) {
            YrTileData td{};
            td.x = tx * ts, td.y = v * r->s.height + ty * ts;
            td.w = std::min(ts, r->s.width - td.x), td.h = std::min(ts, r->s.height - ty * ts);
            td.index = (uint64_t(v) * tilesY + ty) * tilesX + tx, td.total = uint64_t(views) * tilesX * tilesY;
            const double share = double(td.w) * td.h / px;
            td.rays = uint64_t(double(waveRays) * share), td.timeMs = waveMs * share;
            r->tileCb(&data, &td, r->tileUser);
          }
    }
    if (r->cb) {
      YrWaveData wd{wave, waveSamples, waveRays, waveMs};
      r->cb(&data, &wd, r->cbUser);
    }
    raysBefore = agree[0];
    if (r->adaptive && agree[2] == 0) break;  // every pixel has stopped: the render is complete
    const uint64_t next = (wave > 0 || waveSamples > 1) ? std::min<uint64_t>(waveSamples * 2, maxWave) : 1;
    waveSamples = std::min<uint64_t>(next, remaining);
    wave++;
  }
  if (r->aovs && r->comm) {
    // tile sharding (bucket sharding refuses AOVs): the shards' planes into the root's, once per render — after an abort
    // too, since the abort vote has brought every participant here
    rc = onShards(r, [&](size_t i) { return yc_comm_reduce_aovs(r->shards[i].ctx, 0); });
    if (rc != YC_OK) return rfail(r, rc, r->err);
  }
  if (r->adaptive && r->comm) {  // the same for the adaptive planes (bucket sharding refuses adaptive sampling)
    rc = onShards(r, [&](size_t i) { return yc_comm_reduce_adaptive(r->shards[i].ctx, 0); });
    if (rc != YC_OK) return rfail(r, rc, r->err);
  }
  {
    std::lock_guard<std::mutex> lk(r->m);
    r->last = data;
  }
  if (out) *out = data;
  if (r->doneCb) r->doneCb(&data, aborted ? 1 : 0, r->doneUser);  // onRenderAborted / onRenderComplete
  return aborted ? YC_ERR_ABORTED : YC_OK;
}

extern "C" int yr_render_sync(yr_renderer* r, YrRenderData* out) {
  if (!r) return YC_ERR_INVALID;
  if (r->worker.joinable()) r->worker.join();
  r->stop = 0;
  r->running = true;
  r->lastRc = renderBlocking(r, out);
  r->running = false;
  return r->lastRc;
}

extern "C" int yr_render(yr_renderer* r) {
  if (!r) return YC_ERR_INVALID;
  r->stop = 1;  // Renderer::render aborts a render in progress first (tile-renderer.hpp:40-43)
  if (r->worker.joinable()) r->worker.join();
  r->stop = 0;
  r->running = true;
  r->worker = std::thread([r] {
    r->lastRc = renderBlocking(r, nullptr);
    r->running = false;
  });
  return YC_OK;
}

// Renderer::abort(): returns at once; the render stops at its next chunk or bounce boundary (the reference stops
// between tiles, tile-renderer.hpp:182-185) and reports through the done callback.  yr_wait joins.
extern "C" int yr_abort(yr_renderer* r) {
  if (!r) return YC_ERR_INVALID;
  r->stop = 1;
  return YC_OK;
}

extern "C" int yr_wait(yr_renderer* r) {
  if (!r) return YC_ERR_INVALID;
  if (r->worker.joinable()) r->worker.join();
  return r->lastRc;
}

extern "C" int yr_write_ppm(yr_renderer* r, const char* path) {
  if (!r || !path) return YC_ERR_INVALID;
  std::vector<float> ldr(size_t(r->s.width) * frameRows(r) * 4);
  int rc = readFrames(r, nullptr, ldr.data());
  if (rc != YC_OK) return rfail(r, rc, yc_last_error(r->shards[0].ctx));
  return writePpm(path, ldr.data(), r->s.width, frameRows(r)) ? YC_OK : rfail(r, YC_ERR_IO, std::string("cannot write ") + path);
}

extern "C" int yr_read(yr_renderer* r, float* hdrRGBA, float* ldrRGBA, YcStats* stats) {
  if (!r) return YC_ERR_INVALID;
  int rc = readFrames(r, hdrRGBA, ldrRGBA);
  if (rc != YC_OK) return rfail(r, rc, yc_last_error(r->shards[0].ctx));
  if (stats) {
    memset(stats, 0, sizeof *stats);
    for (Shard& sh : r->shards) {  // local shards; with one process per GPU these are this rank's own figures
      YcStats st{};
      if ((rc = yc_resolve(sh.ctx, nullptr, nullptr, &st)) != YC_OK) return rfail(r, rc, yc_last_error(sh.ctx));
      stats->raysReference += st.raysReference, stats->raysExtend += st.raysExtend, stats->raysShadow += st.raysShadow;
      stats->kernelLaunches += st.kernelLaunches, stats->boxTests += st.boxTests, stats->triTests += st.triTests;
      stats->gpuMs = std::max(stats->gpuMs, st.gpuMs), stats->extendMs += st.extendMs, stats->extendLaunches += st.extendLaunches;
    }
  }
  return YC_OK;
}

extern "C" int yr_enable_aovs(yr_renderer* r, int enable) {
  if (!r) return YC_ERR_INVALID;
  if (r->running) return rfail(r, YC_ERR_STATE, "yr_enable_aovs while a render runs");
  if (enable && r->s.integrator == YC_INTEGRATOR_NAIVE)
    return rfail(r, YC_ERR_UNSUPPORTED, "AOVs: the naive integrator runs whole paths in one kernel");
  if (enable && r->comm && r->s.sharding == YR_SHARD_BUCKETS)
    return rfail(r, YC_ERR_UNSUPPORTED, "AOVs with bucket sharding: a pixel's samples are split over the participants");
  r->aovs = enable != 0;  // applied to the contexts by the next render's yc_begin_frame
  return YC_OK;
}

extern "C" int yr_read_aovs(yr_renderer* r, float* albedoRGBA, float* normalDepthRGBA) {
  if (!r) return YC_ERR_INVALID;
  if (r->running) return rfail(r, YC_ERR_STATE, "yr_read_aovs while a render runs");
  if (!r->aovs) return rfail(r, YC_ERR_STATE, "yr_read_aovs: AOVs are not enabled (yr_enable_aovs)");
  yc_ctx* c0 = r->shards[0].ctx;
  int rc = YC_OK;
  if (r->comm && r->s.sharding == YR_SHARD_TILES) {
    if (rootHere(r)) rc = yc_resolve_aovs_combined(c0, albedoRGBA, normalDepthRGBA);
  } else {
    rc = yc_resolve_aovs(c0, albedoRGBA, normalDepthRGBA);
  }
  return rc != YC_OK ? rfail(r, rc, yc_last_error(c0)) : YC_OK;
}

extern "C" int yr_set_adaptive(yr_renderer* r, const YcAdaptive* params) {
  if (!r) return YC_ERR_INVALID;
  if (r->running) return rfail(r, YC_ERR_STATE, "yr_set_adaptive while a render runs");
  if (params && !(std::isfinite(params->threshold) && params->threshold >= 0.0f && std::isfinite(params->lumaFloor) &&
                  params->lumaFloor > 0.0f))
    return rfail(r, YC_ERR_INVALID, "yr_set_adaptive: threshold must be finite and >= 0, lumaFloor finite and > 0");
  if (params && r->comm && r->s.sharding == YR_SHARD_BUCKETS)
    return rfail(r, YC_ERR_UNSUPPORTED, "adaptive sampling with bucket sharding: a pixel's samples are split over the participants");
  r->adaptive = params != nullptr;  // applied to the contexts by the next render, after its yc_begin_frame
  if (params) r->adParams = *params;
  return YC_OK;
}

extern "C" int yr_read_adaptive(yr_renderer* r, uint32_t* samples, float* error) {
  if (!r) return YC_ERR_INVALID;
  if (r->running) return rfail(r, YC_ERR_STATE, "yr_read_adaptive while a render runs");
  if (!r->adaptive) return rfail(r, YC_ERR_STATE, "yr_read_adaptive: adaptive sampling is off (yr_set_adaptive)");
  yc_ctx* c0 = r->shards[0].ctx;
  int rc = YC_OK;
  if (r->comm && r->s.sharding == YR_SHARD_TILES) {
    if (rootHere(r)) rc = yc_resolve_adaptive_combined(c0, samples, error);
  } else {
    rc = yc_resolve_adaptive(c0, samples, error, nullptr);
  }
  return rc != YC_OK ? rfail(r, rc, yc_last_error(c0)) : YC_OK;
}

extern "C" const float* ys_lut_tables(size_t* count) {
  static HostScene holder;
  static std::once_flag once;
  std::call_once(once, [] {
    std::string err;
    holder.loadLuts(&err);
  });
  if (count) *count = holder.lutTables.size();
  return holder.lutTables.empty() ? nullptr : holder.lutTables.data();
}
