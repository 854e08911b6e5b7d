// kat.cuh — function-level known-answer hooks (yc_kat).  Included at the end of wavefront.cu.
//
// Each kind evaluates restated device math on caller-supplied inputs so tests can compare it with
// the reference functions run by oracle/ref_driver.cpp `kat <kind>` on the SAME input blob (the
// blob layouts are documented there).  Kinds that need materials / lights / textures use the scene
// uploaded into the context; "camera" uses the context's camera.
#pragma once

namespace {

struct KatIO {
  const uint32_t* in;  // first record (header skipped)
  float* out;
  YB_DEV float f(size_t w) const { return __uint_as_float(in[w]); }
  YB_DEV V3 v3(size_t w) const { return V3(f(w), f(w + 1), f(w + 2)); }
  YB_DEV V2 v2(size_t w) const { return V2(f(w), f(w + 1)); }
};

struct KatSampler {
  KatIO io;
  SamplerConfig cfg;
  YB_DEV void operator()(uint32_t i) const {
    const size_t r = size_t(i) * 3;
    Sampler s;
    s.start(cfg, io.in[r], io.in[r + 1], io.in[r + 2]);
    const V2 a = s.get2D(), b = s.get2D();
    const float c = s.get1D(), d = s.get1D();
    const V2 e = s.get2D();
    float* o = io.out + size_t(i) * 8;
    o[0] = a.x, o[1] = a.y, o[2] = b.x, o[3] = b.y, o[4] = c, o[5] = d, o[6] = e.x, o[7] = e.y;
  }
};

struct KatLut {
  KatIO io;
  const float* lut;
  YB_DEV void operator()(uint32_t i) const {
    const size_t r = size_t(i) * 4;
    const float a = io.f(r), b = io.f(r + 1), c = io.f(r + 2), ior = io.f(r + 3);
    float* o = io.out + size_t(i) * 8;
    o[0] = ggxE(lut, a, b);
    o[1] = ggxEavg(lut, b);
    o[2] = ggxBaseE(lut, a, b, c);
    o[3] = ggxBaseEavg(lut, a, b);
    o[4] = ggxGlassE(lut, ior, b, c);
    o[5] = ggxGlassEavg(lut, ior, b);
    o[6] = fresnelDielectric(a * 2.0f - 1.0f, ior);
    o[7] = roughen(b);
  }
};

struct KatGgx {
  KatIO io;
  YB_DEV void operator()(uint32_t i) const {
    const size_t r = size_t(i) * 10;
    const GGX g(io.f(r), io.f(r + 1));
    const V3 w = io.v3(r + 2), wm = io.v3(r + 5);
    const V2 u = io.v2(r + 8);
    const V3 s = g.sampleVisibleMicrofacet(w, u);
    float* o = io.out + size_t(i) * 8;
    o[0] = g.mdf(wm), o[1] = g.g1(w), o[2] = g.g(w, wm), o[3] = g.vmdf(w, wm), o[4] = g.smooth() ? 1.0f : 0.0f;
    o[5] = s.x, o[6] = s.y, o[7] = s.z;
  }
};

struct KatBsdf {
  KatIO io;
  DScene sc;
  YB_DEV void operator()(uint32_t i) const {
    const size_t r = size_t(i) * 22;
    const YcMaterial& mat = sc.materials[io.in[r]];
    const V3 wo = io.v3(r + 1), wi = io.v3(r + 4), n = io.v3(r + 7), t = io.v3(r + 10);
    const V2 uv = io.v2(r + 13), u = io.v2(r + 15);
    const float uc = io.f(r + 17), uc2 = io.f(r + 18);
    const bool reg = io.in[r + 19] != 0;
    const float tgw = io.f(r + 20), dist = io.f(r + 21);
    const Bsdf b(sc, mat);
    const V3 f = b.f(wo, wi, n, t, uv);
    const float pdf = b.pdf(wo, wi, n, t, uv);
    const BSDFSample s = b.sample(wo, n, t, uv, u, uc, uc2, reg);
    const V3 base = materialBase(sc, mat, uv), nn = shadingNormal(sc, mat, n, t, tgw, uv), att = b.attenuation(dist);
    float* o = io.out + size_t(i) * 27;
    o[0] = f.x, o[1] = f.y, o[2] = f.z, o[3] = pdf;
    o[4] = __uint_as_float(uint32_t(s.scatter));
    o[5] = s.f.x, o[6] = s.f.y, o[7] = s.f.z;
    o[8] = s.Le.x, o[9] = s.Le.y, o[10] = s.Le.z;
    o[11] = s.wi.x, o[12] = s.wi.y, o[13] = s.wi.z;
    o[14] = s.pdf, o[15] = s.roughness;
    o[16] = materialAlpha(sc, mat, uv);
    o[17] = base.x, o[18] = base.y, o[19] = base.z;
    o[20] = __uint_as_float((mat.thinTransmission && mat.transmission > 0.0f) ? 1u : 0u);
    o[21] = nn.x, o[22] = nn.y, o[23] = nn.z;
    o[24] = att.x, o[25] = att.y, o[26] = att.z;
  }
};

struct KatLight {
  KatIO io;
  DScene sc;
  YB_DEV void operator()(uint32_t i) const {
    const size_t r = size_t(i) * 13;
    const uint32_t li = io.in[r];
    const YcLight& L = sc.lights[li];
    const V3 p = io.v3(r + 1);
    const V2 u = io.v2(r + 7);
    const V3 wi = io.v3(r + 9);
    const float uc = io.f(r + 12);
    const LightSample s = lightSample(sc, L, p, u);
    const V3 Le = lightLe(sc, L, octahedralUV(wi));
    const PickedLight pk = pickLight(sc, uc);
    float* o = io.out + size_t(i) * 22;
    o[0] = s.Li.x, o[1] = s.Li.y, o[2] = s.Li.z;
    o[3] = s.wi.x, o[4] = s.wi.y, o[5] = s.wi.z;
    o[6] = s.p.x, o[7] = s.p.y, o[8] = s.p.z;
    o[9] = s.n.x, o[10] = s.n.y, o[11] = s.n.z;
    o[12] = s.pdf;
    o[13] = lightPdf(sc, L, wi);
    o[14] = L.power;
    o[15] = __uint_as_float(L.type == YC_LIGHT_AREA ? 0u : 1u);
    o[16] = Le.x, o[17] = Le.y, o[18] = Le.z;
    o[19] = __uint_as_float(pk.index);
    o[20] = pk.p;
    o[21] = lightPickProbability(sc, li);
  }
};

#ifdef YB_RNG_SAMPLERS
// UniformLightSampler (same input records as KatLight): out = {picked index, pick probability, p(light)}
struct KatLightUniform {
  KatIO io;
  DScene sc;
  YB_DEV void operator()(uint32_t i) const {
    const size_t r = size_t(i) * 13;
    const PickedLight pk = pickLightUniform(sc, io.f(r + 12));
    float* o = io.out + size_t(i) * 3;
    o[0] = __uint_as_float(pk.index);
    o[1] = pk.p;
    o[2] = 1.0f / float(sc.nLights);
  }
};
#endif

struct KatGmon {
  KatIO io;
  uint32_t n;
  YB_DEV void operator()(uint32_t i) const {
    const int m = estimatorBuckets(int(n), kMaxBuckets);
    float* o = io.out + size_t(i) * 9;
    for (int est = 0; est < 3; est++) {  // GMoN, MoN, Mean — the order ref_driver writes them
      V3 acc[kMaxBuckets];
      uint32_t cnt[kMaxBuckets];
      for (int b = 0; b < kMaxBuckets; b++) cnt[b] = 0;
      const int mm = est == YC_ESTIMATOR_MEAN ? 1 : m;
      for (uint32_t s = 0; s < n; s++) {
        const V3 v = io.v3((size_t(i) * n + s) * 3);
        const int b = est == YC_ESTIMATOR_MEAN ? 0 : int(s % uint32_t(mm));
        if (estimatorAccepts(est, v)) {
          acc[b] += v;
          cnt[b]++;
        }
      }
      const V3 val = estimatorValue(est, acc, cnt, mm, n);
      o[est * 3] = val.x, o[est * 3 + 1] = val.y, o[est * 3 + 2] = val.z;
    }
  }
};

// GMoNbEstimator alone (same input as KatGmon): out = value[3]
struct KatGmonb {
  KatIO io;
  uint32_t n;
  YB_DEV void operator()(uint32_t i) const {
    const int m = estimatorBuckets(int(n), kMaxBuckets);
    V3 acc[kMaxBuckets];
    uint32_t cnt[kMaxBuckets];
    for (int b = 0; b < kMaxBuckets; b++) cnt[b] = 0;
    for (uint32_t s = 0; s < n; s++) {
      const V3 v = io.v3((size_t(i) * n + s) * 3);
      if (estimatorAccepts(YC_ESTIMATOR_GMONB, v)) {
        acc[s % uint32_t(m)] += v;
        cnt[s % uint32_t(m)]++;
      }
    }
    const V3 val = estimatorValue(YC_ESTIMATOR_GMONB, acc, cnt, m, n);
    float* o = io.out + size_t(i) * 3;
    o[0] = val.x, o[1] = val.y, o[2] = val.z;
  }
};

struct KatAgx {
  KatIO io;
  uint32_t tonemap;
  YB_DEV void operator()(uint32_t i) const {
    const V3 v = agx(io.v3(size_t(i) * 3), agxLook(tonemap));
    float* o = io.out + size_t(i) * 3;
    o[0] = v.x, o[1] = v.y, o[2] = v.z;
  }
};

struct KatCamera {
  KatIO io;
  YcCamera cam;
  YB_DEV void operator()(uint32_t i) const {
    const size_t r = size_t(i) * 6;
    V3 o, d;
    cameraRay(cam, io.in[r], io.in[r + 1], io.v2(r + 2), io.v2(r + 4), o, d);
    float* out = io.out + size_t(i) * 6;
    out[0] = o.x, out[1] = o.y, out[2] = o.z, out[3] = d.x, out[4] = d.y, out[5] = d.z;
  }
};

struct KatTexture {
  KatIO io;
  DScene sc;
  YB_DEV void operator()(uint32_t i) const {
    const size_t r = size_t(i) * 3;
    const int ti = int(io.in[r]);
    const V2 uv = io.v2(r + 1);
    const YcTexture t = sc.textures[ti];
    float* o = io.out + size_t(i) * 4;
    o[0] = o[1] = o[2] = o[3] = 0.0f;
    if (t.isFloat) {
      const V3 v = sampleHDR(sc, ti, uv);
      o[0] = v.x, o[1] = v.y, o[2] = v.z;
    } else {
      const TexTaps k = texTaps(t, uv);
      for (uint32_t c = 0; c < t.channels; c++) o[c] = sampleU8Channel(sc, t, k, c);
    }
  }
};

}  // namespace

extern "C" int yc_kat(yc_ctx* ctx, const char* kind, const void* in, size_t inBytes, void* out, size_t outBytes) {
  if (!ctx || !kind || !in || !out || inBytes < 4 || (inBytes & 3)) return YC_ERR_INVALID;
  rt::useDevice(ctx->device);
  const std::string k = kind;
  const uint32_t* hin = static_cast<const uint32_t*>(in);
  const size_t inWords = inBytes / 4;
  size_t header = 1, recWords = 0, outWords = 0;
  uint32_t n = hin[0];
  const bool needsScene = k == "bsdf" || k == "light" || k == "lightuniform" || k == "texture" || k == "lut";
  if (needsScene && !ctx->hasScene) return fail(ctx, YC_ERR_NO_SCENE, "yc_kat(%s) needs an uploaded scene", kind);
  if (k == "sampler") header = 2, n = inWords > 1 ? hin[1] : 0, recWords = 3, outWords = 8;
  else if (k == "lut") recWords = 4, outWords = 8;
  else if (k == "ggx") recWords = 10, outWords = 8;
  else if (k == "bsdf") recWords = 22, outWords = 27;
  else if (k == "light") recWords = 13, outWords = 22;
#ifdef YB_RNG_SAMPLERS
  else if (k == "lightuniform") recWords = 13, outWords = 3;
#endif
  else if (k == "gmon") header = 2, n = inWords > 1 ? hin[1] : 0, recWords = size_t(hin[0]) * 3, outWords = 9;
  else if (k == "gmonb") header = 2, n = inWords > 1 ? hin[1] : 0, recWords = size_t(hin[0]) * 3, outWords = 3;
  else if (k == "agx") header = 2, n = inWords > 1 ? hin[1] : 0, recWords = 3, outWords = 3;
  else if (k == "camera") header = 15, n = inWords > 14 ? hin[14] : 0, recWords = 6, outWords = 6;
  else if (k == "texture") recWords = 3, outWords = 4;
  else return fail(ctx, YC_ERR_INVALID, "unknown kat kind %s", kind);
  if (inWords < header + size_t(n) * recWords || outBytes < size_t(n) * outWords * 4)
    return fail(ctx, YC_ERR_INVALID, "yc_kat(%s): buffer sizes do not match %u records", kind, n);
  if (k == "camera" && ctx->cams.empty()) return fail(ctx, YC_ERR_STATE, "yc_kat(camera) needs yc_set_camera");
  if (n == 0) return YC_OK;
  void *din = nullptr, *dout = nullptr;
  YC_TRY(rt::alloc(&din, inBytes));
  const char* e = rt::alloc(&dout, size_t(n) * outWords * 4);
  if (!e) e = rt::h2d(ctx->st, din, in, inBytes);
  if (!e) {
    KatIO io{static_cast<const uint32_t*>(din) + header, static_cast<float*>(dout)};
    if (k == "sampler") {
      SamplerConfig cfg;
      cfg.log2spp = log2IntU(hin[0]);
      cfg.nBase4Digits = 6 + (cfg.log2spp + 1) / 2;  // renderSize {64, 64}
      cfg.scrambler = ctx->opts.scrambler;
      cfg.kind = ctx->opts.sampler;
      cfg.strata = uint32_t(std::ceil(std::sqrt(double(hin[0]))));
      rt::launchFor(ctx->st, n, KatSampler{io, cfg});
    } else if (k == "lut") rt::launchFor(ctx->st, n, KatLut{io, ctx->ds.lut});
    else if (k == "ggx") rt::launchFor(ctx->st, n, KatGgx{io});
    else if (k == "bsdf") rt::launchFor(ctx->st, n, KatBsdf{io, ctx->ds});
    else if (k == "light") rt::launchFor(ctx->st, n, KatLight{io, ctx->ds});
#ifdef YB_RNG_SAMPLERS
    else if (k == "lightuniform") rt::launchFor(ctx->st, n, KatLightUniform{io, ctx->ds});
#endif
    else if (k == "gmon") rt::launchFor(ctx->st, n, KatGmon{io, hin[0]});
    else if (k == "gmonb") rt::launchFor(ctx->st, n, KatGmonb{io, hin[0]});
    else if (k == "agx") rt::launchFor(ctx->st, n, KatAgx{io, hin[0] == 1 ? uint32_t(YC_TONEMAP_AGX_GOLDEN) : hin[0] == 2 ? uint32_t(YC_TONEMAP_AGX_PUNCHY) : uint32_t(YC_TONEMAP_AGX)});
    else if (k == "camera") rt::launchFor(ctx->st, n, KatCamera{io, ctx->cams[0]});
    else rt::launchFor(ctx->st, n, KatTexture{io, ctx->ds});
    ctx->launches++;
    e = rt::d2h(ctx->st, out, dout, size_t(n) * outWords * 4);
    if (!e) e = rt::lastError();
  }
  rt::release(din);
  rt::release(dout);
  if (e) return fail(ctx, YC_ERR_CUDA, "yc_kat(%s): %s", kind, e);
  return YC_OK;
}
