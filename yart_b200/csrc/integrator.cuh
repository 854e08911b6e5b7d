// integrator.cuh — per-path stages of the wavefront MIS+NEE integrator.
//
// One camera path of the reference's MISIntegrator::Li (src/cpu/mis-integrator.cpp:13-106, with Ld
// :111-133 and unoccluded :135-148) is cut into stages that run as separate kernels over queues of
// path indices:
//     raygen   RayIntegrator::sample            ray-integrator.cpp:11-18, integrator.cpp:20
//     extend   testNode (closest hit)           mis-integrator.cpp:26
//     shade    miss/env, BSDF sample, emission, NEE set-up, throughput, next ray, Russian roulette
//                                                mis-integrator.cpp:27-102, 111-124, 128-132
//     shadow   unoccluded() + the L += of Ld    mis-integrator.cpp:79-80, 124-126, 135-148
// Every sampler draw happens in the reference's order (SURVEY Appendix A.1).  Only when the scene
// has alpha-tested materials can traversal consume draws (ray-integrator.cpp:211); then the
// Russian-roulette draw, which follows the shadow ray's draws, is deferred to the head of the next
// extend stage (DEFER_RR) and shadow writes the path's sampler dimension back.
// Additions into L happen in the reference's order (shade(b) → shadow(b) → shade(b+1)), so a path's
// radiance has the same rounding sequence as the oracle's.
#pragma once
#include "camera.cuh"
#include "lights.cuh"
#include "wide_bvh.cuh"

namespace yb {

constexpr uint32_t kFlagDepthMask = 0xffu;
constexpr uint32_t kFlagSpecular = 1u << 8;
constexpr uint32_t kFlagRegularized = 1u << 9;
constexpr uint32_t kFlagPendingRR = 1u << 10;
constexpr int32_t kHitMiss = -1;
constexpr int32_t kHitDead = -2;  // path ended by a deferred Russian roulette: shade must skip it
constexpr uint32_t kBackSideBit = 1u << 30;

// Path state in HBM, SoA over path slots (one slot per pixel-sample of the current chunk).
struct PathState {
  float4* rayO;     // origin.xyz, lastPdf
  float4* rayD;     // dir.xyz, accRoughness
  float4* L;        // radiance.rgb, unused
  float4* att;      // throughput.rgb, unused
  uint32_t* dim;    // sampler dimension
  uint32_t* flags;  // depth | kFlag*
  float4* hitA;     // t, u, v, prim (bits)
  int32_t* hitB;    // node | backSide << 30, or kHitMiss / kHitDead
};

// NEE requests, compacted (one per shadow ray of the current bounce).
struct ShadowQueue {
  float4* o;    // origin.xyz, tMax
  float4* d;    // dir.xyz, |wi . n|
  float4* lif;  // (Li * f).rgb, pdfBSDF + pdfLight
  float4* att;  // path throughput before this bounce's update .rgb, path index (bits)
};

struct Counters {
  unsigned long long raysReference, raysExtend, raysShadow, boxTests, triTests;  // raysExtend: tail kernel only
};

// Everything a stage needs besides the scene.
struct WaveParams {
  YcCamera cam;
  SamplerConfig smp;
  float bg[3];
  uint32_t maxDepth;
  // chunk geometry: path i ↔ pixel pixelList[pixBase + i % nPix], sample s0 + (i / nPix) * (sStrideM1 + 1)
  const uint32_t* pixelList;  // x | y << 16
  uint32_t pixBase, nPix, s0;
  uint32_t sStrideM1;  // sample stride - 1: 0 for consecutive samples, m - 1 when a chunk holds one estimator bucket's samples
};

YB_DEV void pathPixelSample(const WaveParams& w, uint32_t i, uint32_t& px, uint32_t& py, uint32_t& sample) {
  const uint32_t pix = w.pixelList[w.pixBase + i % w.nPix];
  px = pix & 0xffffu;
  py = pix >> 16;
  sample = w.s0 + (i / w.nPix) * (w.sStrideM1 + 1u);
}

YB_DEV Sampler pathSampler(const WaveParams& w, uint32_t i, uint32_t dim) {
  uint32_t px, py, s;
  pathPixelSample(w, i, px, py, s);
  Sampler smp;
  smp.start(w.smp, px, py, s);
  smp.dim = dim;
  return smp;
}

// ---- raygen ---------------------------------------------------------------------------
YB_DEV void raygenStage(const WaveParams& w, const PathState& ps, uint32_t i) {
  uint32_t px, py, s;
  pathPixelSample(w, i, px, py, s);
  Sampler smp;
  smp.start(w.smp, px, py, s);  // Integrator::render, integrator.cpp:20
  V3 o, d;
  primaryRay(w.cam, smp, px, py, o, d);
  ps.rayO[i] = make_float4(o.x, o.y, o.z, 0.0f);
  ps.rayD[i] = make_float4(d.x, d.y, d.z, 0.0f);
  ps.L[i] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
  ps.att[i] = make_float4(1.0f, 1.0f, 1.0f, 0.0f);
  ps.dim[i] = smp.dim;
  ps.flags[i] = 0u;
}

// Russian roulette, mis-integrator.cpp:97-102.  Returns false when the path dies.
YB_DEV bool russianRoulette(Sampler& smp, uint32_t depth, V3& att) {
  if (depth > 1 && maxComponent(att) < 1.0f) {
    const float a = 1.0f - maxComponent(att);
    const float q = 0.0f < a ? a : 0.0f;  // std::max(0.0f, a)
    if (smp.get1D() < q) return false;
    att /= 1.0f - q;
  }
  return true;
}

// ---- extend ---------------------------------------------------------------------------
// ALPHA: scene has alpha-tested materials (traversal draws from the path's sampler).
// extendLoad / extendStore bracket the closest-hit traversal of one path, so the sequential driver
// below and the persistent warp kernel (trace_kernels.cuh) share every bit of arithmetic.
template <bool ALPHA>
YB_DEV bool extendLoad(const WaveParams& w, const PathState& ps, uint32_t i, V3& o, V3& d, Sampler& smp) {
  const float4 ro = ps.rayO[i], rd = ps.rayD[i];
  o = V3(ro.x, ro.y, ro.z);
  d = V3(rd.x, rd.y, rd.z);
  if (ALPHA) {
    smp = pathSampler(w, i, ps.dim[i]);
    const uint32_t fl = ps.flags[i];
    if (fl & kFlagPendingRR) {
      const float4 a4 = ps.att[i];
      V3 att(a4.x, a4.y, a4.z);
      const uint32_t depth = fl & kFlagDepthMask;
      const bool alive = russianRoulette(smp, depth, att) && depth < w.maxDepth;
      ps.flags[i] = fl & ~kFlagPendingRR;
      ps.dim[i] = smp.dim;
      if (!alive) {
        ps.hitB[i] = kHitDead;
        return false;
      }
      ps.att[i] = make_float4(att.x, att.y, att.z, 0.0f);
    }
  }
  return true;
}

template <bool ALPHA>
YB_DEV void extendStore(const PathState& ps, uint32_t i, const TraceState& st, const Sampler& smp) {
  if (ALPHA) ps.dim[i] = smp.dim;
  ps.hitA[i] = make_float4(st.hit.t, st.hit.u, st.hit.v, __uint_as_float(st.hit.prim));
  ps.hitB[i] = st.hit.node < 0 ? kHitMiss : int32_t(uint32_t(st.hit.node) | (st.hit.backSide ? kBackSideBit : 0u));
}

YB_DEV void initTraceState(TraceState& st, float tMax) {
  st.hit.t = tMax;
  st.hit.u = st.hit.v = 0.0f;
  st.hit.prim = 0xffffffffu;
  st.hit.node = kHitMiss;
  st.hit.backSide = 0;
  st.attenuation = V3(1.0f);
}

// Walk: the BVH layout, Bvh2Walk (reference order, traverse.cuh) or WideWalk (the collapsed 4-wide BVH, wide_bvh.cuh;
// scenes without alpha-tested materials only).
template <bool ALPHA, bool COUNT, class Walk = Bvh2Walk>
YB_DEV void extendStage(const DScene& sc, const WaveParams& w, const PathState& ps, uint32_t i, TravStack& stack,
                        TraceCounters& cnt) {
  V3 o, d;
  Sampler smp;
  if (!extendLoad<ALPHA>(w, ps, i, o, d, smp)) return;
  TraceState st;
  initTraceState(st, INFINITY);
  traceScene<Walk, false, ALPHA, COUNT, false>(sc, o, d, st, stack, &smp, cnt);
  extendStore<ALPHA>(ps, i, st, smp);
}

// ---- shade ----------------------------------------------------------------------------
struct ShadowRequest {
  V3 o, d, lif, att;
  float tMax, absDotN, denom;
};

enum : uint32_t { kShadeContinue = 1u, kShadeShadow = 2u };

// Returns kShade* bits; `rq` is filled when kShadeShadow is set.  DEFER_RR ⇔ scene has alpha.
// Miss shading (mis-integrator.cpp:27-43) as its own stage: extend sorts queue entries into a "hit" and a
// "miss" queue, so the heavy surface-shading code runs in warps where every lane has work.
YB_DEV void shadeMissStage(const DScene& sc, const WaveParams& w, const PathState& ps, uint32_t i, uint32_t& raysReference) {
  raysReference += 1;  // mis-integrator.cpp:22
  const float4 ro4 = ps.rayO[i], rd4 = ps.rayD[i], L4 = ps.L[i], a4 = ps.att[i];
  const V3 rayD(rd4.x, rd4.y, rd4.z);
  const float lastPdf = ro4.w;
  V3 L(L4.x, L4.y, L4.z), att(a4.x, a4.y, a4.z);
  const uint32_t fl = ps.flags[i];
  const uint32_t depth = fl & kFlagDepthMask;
  const bool specularBounce = (fl & kFlagSpecular) != 0;
  // Le(octahedralUV(ray.dir)) ignores the light's transform (SURVEY Appendix A.9)
  for (uint32_t k = 0; k < sc.nInf; k++) {
    const YcLight& light = sc.lights[sc.infLights[k]];
    const V3 Le = lightLe(sc, light, octahedralUV(rayD));
    if (depth == 0 || specularBounce) {
      L += att * Le;
    } else {
      const float pdfLight = lightPdf(sc, light, rayD);
      const float wBSDF = lastPdf / (lastPdf + pdfLight);
      L += att * wBSDF * Le;
    }
  }
  L += att * V3(w.bg);
  ps.L[i] = make_float4(L.x, L.y, L.z, 0.0f);
}

// Surface shading is cut in three so that each kernel's instruction footprint stays near the instruction cache and its
// register need matches what it does (one fused kernel touched 134 KB of SASS per launch and stalled on instruction
// fetch more than on anything else; surface + NEE in two kernels still spilled 1-2 KB per thread at any occupancy that
// hid the gather chain's latency):
//   resolveSurface  the gather chain: hit → node → mesh → indices → vertices → material → texels, the shading frame
//                   (ray-integrator.cpp:56-82, 205-227; core/bsdf.cpp:43-58; parametric.cpp's texture preambles) —
//                   memory latency, few registers, runs at full occupancy — into a SurfRecord;
//   sampleSurface   the BSDF sample, emission MIS, throughput, next ray, Russian roulette (mis-integrator.cpp:46-73,
//                   83-102) from that record — arithmetic only;
//   shadeNee        Ld up to the shadow ray (mis-integrator.cpp:79-80 → :111-124, 135-148) from the same record.
// The sampler dimensions of the NEE draws are reserved by sampleSurface (they precede the roulette draw), so the three
// pieces draw exactly what the fused loop drew; L is only touched by sampleSurface (emission) and later by the shadow
// stage, in the reference's order.
struct SurfRecord {
  V3 p, n, fx, fy;  // hit point, shading normal (= frame z), frame x / y
  V3 woLocal;       // outgoing direction in the frame
  MatEval me;       // material parameters with their textures applied
  V2 uv;
  float t;          // hit distance (volume attenuation, parametric.cpp:834-838)
  int32_t material, lightIdx;
  uint32_t backSide;
};

// SoA storage of SurfRecords, one slot per entry of the bounce's hit queue (7 x float4 = 112 B), plus what
// sampleSurface hands to shadeNee for the hits that take a NEE sample: the throughput before this bounce's update and
// the sampler dimension of the first NEE draw (r7).
struct SurfState {
  float4 *r0, *r1, *r2, *r3, *r4, *r5, *r6, *r7;
};
YB_DEV void storeSurf(const SurfState& ss, uint32_t j, const SurfRecord& r) {
  ss.r0[j] = make_float4(r.p.x, r.p.y, r.p.z, __uint_as_float(uint32_t(r.material) | (r.backSide << 31)));
  ss.r1[j] = make_float4(r.n.x, r.n.y, r.n.z, r.t);
  ss.r2[j] = make_float4(r.fx.x, r.fx.y, r.fx.z, r.me.r);
  ss.r3[j] = make_float4(r.fy.x, r.fy.y, r.fy.z, r.me.m);
  ss.r4[j] = make_float4(r.woLocal.x, r.woLocal.y, r.woLocal.z, r.me.t);
  ss.r5[j] = make_float4(r.me.base.x, r.me.base.y, r.me.base.z, r.me.c);
  ss.r6[j] = make_float4(r.uv.x, r.uv.y, r.me.cr, __uint_as_float(uint32_t(r.lightIdx)));
}
YB_DEV SurfRecord loadSurf(const SurfState& ss, uint32_t j) {
  const float4 a = ss.r0[j], b = ss.r1[j], c = ss.r2[j], d = ss.r3[j], e = ss.r4[j], f = ss.r5[j], g = ss.r6[j];
  SurfRecord r;
  const uint32_t mb = __float_as_uint(a.w);
  r.p = V3(a.x, a.y, a.z), r.material = int32_t(mb & 0x7fffffffu), r.backSide = mb >> 31;
  r.n = V3(b.x, b.y, b.z), r.t = b.w;
  r.fx = V3(c.x, c.y, c.z), r.me.r = c.w;
  r.fy = V3(d.x, d.y, d.z), r.me.m = d.w;
  r.woLocal = V3(e.x, e.y, e.z), r.me.t = e.w;
  r.me.base = V3(f.x, f.y, f.z), r.me.c = f.w;
  r.uv = V2(g.x, g.y), r.me.cr = g.z, r.lightIdx = int32_t(__float_as_uint(g.w));
  return r;
}

enum : uint32_t { kShadeNee = 4u };  // sampleSurface: the bounce takes a NEE sample, run shadeNee on its record

YB_DEV SurfRecord resolveSurface(const DScene& sc, const PathState& ps, uint32_t i) {
  const int32_t hb = ps.hitB[i];
  const float4 ro4 = ps.rayO[i], rd4 = ps.rayD[i];
  const V3 rayO(ro4.x, ro4.y, ro4.z), rayD(rd4.x, rd4.y, rd4.z);
  HitRec h;
  const float4 ha = ps.hitA[i];
  h.t = ha.x, h.u = ha.y, h.v = ha.z, h.prim = __float_as_uint(ha.w);
  h.node = int32_t(uint32_t(hb) & ~kBackSideBit);
  h.backSide = (uint32_t(hb) & kBackSideBit) ? 1u : 0u;
  const SurfaceHit hit = resolveHit(sc, h, rayO, rayD);
  // BSDF::sample / f / pdf (core/bsdf.cpp:5-41) each rebuild the same local frame and re-read the same
  // texels; here they are evaluated once per hit and shared (identical values, see bsdf.cuh).
  const Frame fr = Bsdf::localFrame(hit.n, hit.tg);
  SurfRecord s;
  s.me = evalMaterialTextures(sc, sc.materials[hit.material], hit.uv);
  s.p = hit.p, s.n = hit.n, s.fx = fr.x, s.fy = fr.y;
  s.woLocal = fr.wtl(-rayD);
  s.uv = hit.uv, s.t = h.t;
  s.material = hit.material, s.lightIdx = hit.lightIdx, s.backSide = h.backSide;
  return s;
}

// Returns kShadeContinue / kShadeNee bits; with kShadeNee, `neeAtt` / `neeDim` are what shadeNee needs besides the
// record.  DEFER_RR ⇔ scene has alpha.
template <bool DEFER_RR>
YB_DEV uint32_t sampleSurface(const DScene& sc, const WaveParams& w, const PathState& ps, uint32_t i, const SurfRecord& s,
                              V3& neeAtt, uint32_t& neeDim, uint32_t& raysReference) {
  raysReference += 1;  // mis-integrator.cpp:22
  const float4 ro4 = ps.rayO[i], rd4 = ps.rayD[i], L4 = ps.L[i], a4 = ps.att[i];
  const V3 rayO(ro4.x, ro4.y, ro4.z), rayD(rd4.x, rd4.y, rd4.z);
  float lastPdf = ro4.w, accRoughness = rd4.w;
  V3 L(L4.x, L4.y, L4.z), att(a4.x, a4.y, a4.z);
  uint32_t fl = ps.flags[i];
  uint32_t depth = fl & kFlagDepthMask;
  const bool specularBounce = (fl & kFlagSpecular) != 0, regularized = (fl & kFlagRegularized) != 0;
  const YcMaterial& mat = sc.materials[s.material];
  const Bsdf bsdf(sc, mat);
  Sampler smp = pathSampler(w, i, ps.dim[i]);
  const V3 wo = -rayD;
  Frame fr;
  fr.x = s.fx, fr.y = s.fy, fr.z = s.n;

  // mis-integrator.cpp:46-58
  const V2 u = smp.get2D();
  const float uc = smp.get1D();
  const float uc2 = smp.get1D();
  BSDFSample res = bsdf.sampleImpl(s.woLocal, s.uv, s.me, u, uc, uc2, regularized);
  res.wi = fr.ltw(res.wi);

  // mis-integrator.cpp:61-73 (lastHit.p is this ray's origin: ray = Ray(hit.p, wi), lastHit = hit)
  if (res.is(Emitted)) {
    if (depth == 0 || specularBounce) {
      L += att * res.Le;
    } else if (s.lightIdx != -1) {
      const YcLight& light = sc.lights[s.lightIdx];
      const float pdfLight = lightPdf(sc, light, wo) * length2(rayO - s.p) *
                             lightPickProbability(sc, uint32_t(s.lightIdx)) / absDot(wo, s.n);
      const float wBSDF = lastPdf / (lastPdf + pdfLight);
      L += att * wBSDF * res.Le;
    }
  }

  uint32_t result = 0u;
  if (res.is(Reflected | Transmitted)) {
    // mis-integrator.cpp:79-80 → Ld: its three draws (get1D, get2D) come next in the sampler's order
    if (!res.is(Emitted | Specular) && sc.nLights != 0) {
      neeAtt = att;
      neeDim = smp.dim;
      smp.dim += 3;
      result |= kShadeNee;
    }
    // mis-integrator.cpp:83-95
    const V3 fcos = res.f * absDot(res.wi, s.n);
    att *= fcos / res.pdf;
    if (s.backSide) att *= bsdf.attenuation(s.t);
    fl = 0u;
    if (res.is(Specular)) fl |= kFlagSpecular;
    accRoughness += res.roughness;
    if (accRoughness > 0.5f) fl |= kFlagRegularized;
    lastPdf = res.pdf;
    depth++;
    bool alive = true;
    if (DEFER_RR) {
      fl |= kFlagPendingRR;
      // a path at maxDepth still owes its roulette draw to nobody: the loop ends either way
      alive = depth < w.maxDepth;
    } else {
      alive = russianRoulette(smp, depth, att) && depth < w.maxDepth;
    }
    if (alive) {
      ps.rayO[i] = make_float4(s.p.x, s.p.y, s.p.z, lastPdf);
      ps.rayD[i] = make_float4(res.wi.x, res.wi.y, res.wi.z, accRoughness);
      ps.att[i] = make_float4(att.x, att.y, att.z, 0.0f);
      ps.flags[i] = fl | (depth & kFlagDepthMask);
      result |= kShadeContinue;
    }
  }
  ps.dim[i] = smp.dim;
  ps.L[i] = make_float4(L.x, L.y, L.z, 0.0f);
  return result;
}

// Ld (mis-integrator.cpp:111-133) up to the shadow ray.  Returns true when `rq` holds a request.
YB_DEV bool shadeNee(const DScene& sc, const WaveParams& w, uint32_t i, const SurfRecord& s, V3 att, uint32_t dim,
                     ShadowRequest& rq) {
  const Bsdf bsdf(sc, sc.materials[s.material]);
  Frame fr;
  fr.x = s.fx, fr.y = s.fy, fr.z = s.n;
  Sampler smp = pathSampler(w, i, dim);
  const float ucl = smp.get1D();
  const V2 ul = smp.get2D();
  const PickedLight pick = pickLight(sc, ucl);
  const YcLight& light = sc.lights[pick.index];
  const LightSample ls = lightSample(sc, light, s.p, ul);
  const V3 wiLocal = fr.wtl(ls.wi);
  const V3 f = bsdf.fImpl(s.woLocal, wiLocal, s.me);
  if (length2(f) == 0.0f) return false;
  // unoccluded(), :135-148
  const V3 to = ls.p - s.p;
  rq.o = s.p;
  rq.d = normalized(to);
  rq.tMax = length(to) - 0.001f;
  const float pdfBSDF = bsdf.pdfImpl(s.woLocal, wiLocal, s.me);
  float pdfLight = pick.p * ls.pdf / absDot(ls.n, ls.wi);
  if (light.type == YC_LIGHT_AREA) pdfLight *= length2(s.p - ls.p);
  rq.lif = ls.Li * f;
  rq.absDotN = absDot(ls.wi, s.n);
  rq.denom = pdfBSDF + pdfLight;
  rq.att = att;
  return true;
}

// The three pieces back to back (the per-path tail kernel).  Returns kShade* bits; `rq` is filled when kShadeShadow is set.
template <bool DEFER_RR>
YB_DEV uint32_t shadeStage(const DScene& sc, const WaveParams& w, const PathState& ps, uint32_t i, ShadowRequest& rq,
                           uint32_t& raysReference) {
  const int32_t hb = ps.hitB[i];
  if (hb == kHitDead) return 0u;
  if (hb == kHitMiss) {
    shadeMissStage(sc, w, ps, i, raysReference);
    return 0u;
  }
  const SurfRecord s = resolveSurface(sc, ps, i);
  V3 neeAtt;
  uint32_t neeDim = 0;
  uint32_t result = sampleSurface<DEFER_RR>(sc, w, ps, i, s, neeAtt, neeDim, raysReference);
  if ((result & kShadeNee) && shadeNee(sc, w, i, s, neeAtt, neeDim, rq)) result |= kShadeShadow;
  return result & (kShadeContinue | kShadeShadow);
}

// ---- NaiveIntegrator ------------------------------------------------------------------
// src/cpu/naive-integrator.cpp:12-60: no NEE, no MIS, no Russian roulette.  The reference recurses,
//     Li(depth) = [Le] + Li(depth + 1) * fcos / pdf,
// i.e. the products are formed on the way BACK from the deepest segment, which does not round like a
// forward throughput product.  One thread walks the whole path, records (Le, fcos, pdf) per segment and
// folds them in the recursion's order.  Off the measured path: simplicity over speed.
constexpr uint32_t kNaiveMaxSegments = 64;  // maxDepth + 1 segments at most (`depth > m_maxDepth` ends the path)

template <bool ALPHA>
YB_DEV void naiveStage(const DScene& sc, const WaveParams& w, const PathState& ps, uint32_t i, TravStack& stack,
                       TraceCounters& cnt, uint32_t& raysReference) {
  V3 segLe[kNaiveMaxSegments], segFcos[kNaiveMaxSegments];
  float segPdf[kNaiveMaxSegments];
  uint8_t segFlags[kNaiveMaxSegments];  // 1: emitted, 2: scattered
  uint32_t n = 0;
  V3 tail;  // what the deepest call returns
  for (uint32_t depth = 0;; depth++) {
    if (depth > w.maxDepth || n == kNaiveMaxSegments) break;  // naive-integrator.cpp:21 (returns {})
    raysReference += 1;                                       // :22
    extendStage<ALPHA, false>(sc, w, ps, i, stack, cnt);      // :25 testNode
    const int32_t hb = ps.hitB[i];
    const float4 ro4 = ps.rayO[i], rd4 = ps.rayD[i];
    const V3 rayO(ro4.x, ro4.y, ro4.z), rayD(rd4.x, rd4.y, rd4.z);
    if (hb == kHitMiss) {
      // :26-38 (Le(octahedralUV(ray.dir)) of every infinite light, then the background colour)
      V3 L;
      for (uint32_t k = 0; k < sc.nInf; k++) L += lightLe(sc, sc.lights[sc.infLights[k]], octahedralUV(rayD));
      L += V3(w.bg);
      tail = L;
      break;
    }
    HitRec h;
    const float4 ha = ps.hitA[i];
    h.t = ha.x, h.u = ha.y, h.v = ha.z, h.prim = __float_as_uint(ha.w);
    h.node = int32_t(uint32_t(hb) & ~kBackSideBit);
    h.backSide = (uint32_t(hb) & kBackSideBit) ? 1u : 0u;
    const SurfaceHit hit = resolveHit(sc, h, rayO, rayD);
    const YcMaterial& mat = sc.materials[hit.material];
    const Bsdf bsdf(sc, mat);
    Sampler smp = pathSampler(w, i, ps.dim[i]);
    // :40-48 hit.bsdf->sample(-ray.dir, n, tg, uv, get2D(), get1D(), get1D()) — BSDF::sample, core/bsdf.cpp:27-41.
    // The three draws are function ARGUMENTS, so their order is the compiler's: g++ on x86-64 (the oracle
    // build) evaluates them right to left — uc2 first, then uc, then u — and that is the order kept here
    // (clang evaluates left to right; the reference's source does not pin it).
    const float uc2 = smp.get1D();
    const float uc = smp.get1D();
    const V2 u = smp.get2D();
    ps.dim[i] = smp.dim;
    const Frame fr = Bsdf::localFrame(hit.n, hit.tg);
    const MatEval me = evalMaterialTextures(sc, mat, hit.uv);
    BSDFSample res = bsdf.sampleImpl(fr.wtl(-rayD), hit.uv, me, u, uc, uc2, false);
    res.wi = fr.ltw(res.wi);
    uint8_t fl = 0;
    if (res.is(Emitted)) fl |= 1, segLe[n] = res.Le;  // :51-53
    const bool scattered = res.is(Reflected | Transmitted);
    if (scattered) {
      // :54-59
      fl |= 2;
      segFcos[n] = res.f * absDot(res.wi, hit.n);
      segPdf[n] = res.pdf;
      ps.rayO[i] = make_float4(hit.p.x, hit.p.y, hit.p.z, 0.0f);
      ps.rayD[i] = make_float4(res.wi.x, res.wi.y, res.wi.z, 0.0f);
    }
    segFlags[n++] = fl;
    if (!scattered) break;  // tail stays {}: nothing is added below this segment
  }
  V3 L = tail;
  for (uint32_t k = n; k-- > 0;) {
    V3 Li;
    if (segFlags[k] & 1) Li += segLe[k];
    if (segFlags[k] & 2) Li += L * segFcos[k] / segPdf[k];
    L = Li;
  }
  ps.L[i] = make_float4(L.x, L.y, L.z, 0.0f);
}

// ---- shadow ---------------------------------------------------------------------------
template <bool ALPHA>
YB_DEV uint32_t shadowLoad(const WaveParams& w, const PathState& ps, const ShadowQueue& q, uint32_t j, V3& o, V3& d,
                           float& tMax, Sampler& smp) {
  const float4 o4 = q.o[j], d4 = q.d[j];
  const uint32_t i = __float_as_uint(q.att[j].w);
  o = V3(o4.x, o4.y, o4.z);
  d = V3(d4.x, d4.y, d4.z);
  tMax = o4.w;
  if (ALPHA) smp = pathSampler(w, i, ps.dim[i]);
  return i;
}

// Returns 1 if the NEE sample contributed (the ray the reference counts, mis-integrator.cpp:126).
template <bool ALPHA>
YB_DEV uint32_t shadowFinish(const PathState& ps, const ShadowQueue& q, uint32_t j, uint32_t i, const TraceState& st,
                             bool occluded, const Sampler& smp) {
  if (ALPHA) ps.dim[i] = smp.dim;
  if (occluded) return 0u;
  const float4 l4 = q.lif[j], a4 = q.att[j];
  // Ld: ls.Li * f * att * |wi.n| / (pdfBSDF + pdfLight) (mis-integrator.cpp:132), then L += attenuation * Ld (:80)
  const V3 Ld = V3(l4.x, l4.y, l4.z) * st.attenuation * q.d[j].w / l4.w;
  const float4 L4 = ps.L[i];
  V3 L(L4.x, L4.y, L4.z);
  L += V3(a4.x, a4.y, a4.z) * Ld;
  ps.L[i] = make_float4(L.x, L.y, L.z, 0.0f);
  return 1u;
}

// Without alpha-tested materials nothing observable depends on what an occluded NEE ray finds
// after its first occluder, so the any-hit walk may stop there (EARLY_OUT = !ALPHA); with them the
// sampler draws must match the reference's, which keeps walking (ray-integrator.cpp:121).
template <bool ALPHA, bool COUNT, class Walk = Bvh2Walk>
YB_DEV uint32_t shadowStage(const DScene& sc, const WaveParams& w, const PathState& ps, const ShadowQueue& q,
                            uint32_t j, TravStack& stack, TraceCounters& cnt) {
  V3 o, d;
  float tMax;
  Sampler smp;
  const uint32_t i = shadowLoad<ALPHA>(w, ps, q, j, o, d, tMax, smp);
  TraceState st;
  initTraceState(st, tMax);
  const bool occluded = traceScene<Walk, true, ALPHA, COUNT, !ALPHA>(sc, o, d, st, stack, &smp, cnt);
  return shadowFinish<ALPHA>(ps, q, j, i, st, occluded, smp);
}

}  // namespace yb
