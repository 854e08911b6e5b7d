// traverse.cuh — scene-graph + BVH2 traversal and ray/triangle intersection on the device.
//
// Restates, operation for operation, the reference's
//   RayIntegrator::testNode        src/cpu/ray-integrator.cpp:20-54   (scene graph, node AABB cull)
//   RayIntegrator::testBVH         src/cpu/ray-integrator.cpp:84-160  (stack traversal, near child first)
//   RayIntegrator::testTriangle    src/cpu/ray-integrator.cpp:163-229 (Möller–Trumbore, alpha, NEE transparency)
//   RayIntegrator::testBoundingBox src/cpu/ray-integrator.cpp:231-261 (slab test, two roundings, NaN-tolerant)
//   Ray::Ray                       src/core/ray.hpp:16-26
// The same boxes are tested in the same order with the same arithmetic, so accepted hits (and the
// order of alpha-test sampler draws) are the reference's.  Layout differences only: an inner node
// carries both children's boxes (one 64-B record per visit), leaves are contiguous runs of
// pre-gathered triangles, and the traversal stack lives in shared memory (first kShStack
// entries, one column per thread) with a local-memory spill for deeper trees.
//
// Bvh2Walk is this layout as the scene walks see it (traceScene here, tracePersistent in trace_kernels.cuh);
// WideWalk (wide_bvh.cuh) is the 4-wide one.
#pragma once
#include "sampler.cuh"
#include "scene_dev.cuh"
#include "texture.cuh"

namespace yb {

#ifndef YB_SH_STACK
#define YB_SH_STACK 24
#endif
constexpr int kShStack = YB_SH_STACK;   // shared-memory stack entries per thread
constexpr int kMaxStack = 64;  // reference: stack[64], ray-integrator.cpp:92-93
constexpr float kTMin = 0.001f;

struct TraceCounters {
  uint32_t box = 0, tri = 0;
};

struct LocalRay {
  V3 o, d, idir, odir;
  // ray.hpp:16-26
  YB_DEV void set(V3 origin, V3 dir) {
    o = origin;
    d = dir;
    idir = V3(1.0f / dir.x, 1.0f / dir.y, 1.0f / dir.z);  // 1.0 / dir in double then float ≡ IEEE float divide
    odir = (-origin) / dir;
  }
};

// ray-integrator.cpp:231-261.  lo/hi are the box corners; sign picks per axis.
template <bool COUNT>
YB_DEV bool slab(const LocalRay& r, V3 lo, V3 hi, float tmn, float tmx, float& d, TraceCounters& cnt) {
  if (COUNT) cnt.box++;
  const bool sx = r.d.x < 0.0f, sy = r.d.y < 0.0f, sz = r.d.z < 0.0f;
  V3 bmin(sx ? hi.x : lo.x, sy ? hi.y : lo.y, sz ? hi.z : lo.z);
  V3 bmax(sx ? lo.x : hi.x, sy ? lo.y : hi.y, sz ? lo.z : hi.z);
  V3 tmin = bmin * r.idir + r.odir;  // vec fma(): a*b + c, two roundings (vec.hpp:325-334)
  V3 tmax = bmax * r.idir + r.odir;
  float t0 = tmn, t1 = tmx;
  t0 = rmax(tmin.x, t0);
  t0 = rmax(tmin.y, t0);
  t0 = rmax(tmin.z, t0);
  t1 = rmin(tmax.x, t1);
  t1 = rmin(tmax.y, t1);
  t1 = rmin(tmax.z, t1);
  d = t0;
  return t1 >= t0;
}

// The same test for BVH child boxes inside a live traversal step (hit.t is not NaN there, because a
// step only runs when `d < hit.t` held): with a non-NaN second operand `m > n ? m : n` equals
// fmaxf(m, n) and `m < n ? m : n` equals fminf(m, n) for every m including NaN (both return n), up to
// the sign of a zero that can never be selected (t0 >= tMin > 0) or never matters (t1 = ±0 < t0).
// One FMNMX instead of FSETP + FSEL per fold.
YB_DEV bool slabLive(const LocalRay& r, V3 lo, V3 hi, float tmn, float tmx, float& d) {
  const bool sx = r.d.x < 0.0f, sy = r.d.y < 0.0f, sz = r.d.z < 0.0f;
  V3 bmin(sx ? hi.x : lo.x, sy ? hi.y : lo.y, sz ? hi.z : lo.z);
  V3 bmax(sx ? lo.x : hi.x, sy ? lo.y : hi.y, sz ? lo.z : hi.z);
  V3 tmin = bmin * r.idir + r.odir;
  V3 tmax = bmax * r.idir + r.odir;
  const float t0 = fmaxf(tmin.z, fmaxf(tmin.y, fmaxf(tmin.x, tmn)));
  const float t1 = fminf(tmax.z, fminf(tmax.y, fminf(tmax.x, tmx)));
  d = t0;
  return t1 >= t0;
}

// Per-thread traversal stack: column `tid` of two shared arrays + local spill.
struct TravStack {
  uint32_t* shRef;
  float* shD;
  uint32_t stride;
  uint32_t spillRef[kMaxStack - kShStack];
  float spillD[kMaxStack - kShStack];
  YB_DEV void push(int sp, uint32_t ref, float d) {
    if (sp < kShStack) {
      shRef[sp * stride] = ref;
      shD[sp * stride] = d;
    } else if (sp < kMaxStack) {
      spillRef[sp - kShStack] = ref;
      spillD[sp - kShStack] = d;
    }
  }
  YB_DEV void pop(int sp, uint32_t& ref, float& d) const {
    if (sp < kShStack) {
      ref = shRef[sp * stride];
      d = shD[sp * stride];
    } else {
      ref = spillRef[sp - kShStack];
      d = spillD[sp - kShStack];
    }
  }
};

#ifndef YB_HOSTSIM
constexpr int kTraceBlock = 128;       // 4 warps per CTA of the persistent kernels (trace_kernels.cuh)

// Scheduling knobs (they change only how lanes are grouped, never a ray's own test sequence).
struct TraceTuning {
  int refillMin;  // refill the warp from the queue when at least this many lanes are idle
  int innerMin;   // keep stepping inner nodes while at least this many lanes sit on one
  int shEntries;  // shared-memory stack entries in use (2..kPsStack; the rest spills): tests shrink it to exercise the spill path
};

// Per-lane traversal stack of the persistent kernels: packed (ref, d) entries, [entry][thread] in shared
// memory (one 64-bit access per push / pop, conflict-free), global spill area beyond kPsStack entries.
// The stack pointer is the shared-memory byte address of the next free slot, so push / pop are one
// add and one LDS.64 / STS.64; entry 0 holds a sentinel (kNoRef) written when a mesh is entered, so a
// pop never tests for "empty": popping the sentinel yields kNoRef = "this mesh is walked".
constexpr int kPsStack = kShStack + 1;
constexpr uint32_t kPsStride = kTraceBlock * 8;  // bytes between consecutive entries of one thread
constexpr int kSpillEntries = kMaxStack;         // global spill entries per thread (covers the smallest shared stack)
constexpr uint32_t kNoRef = 0xffffffffu;   // "no current node" (has the leaf bit: never stepped as inner)
constexpr uint32_t kPopRef = 0xfffffffeu;  // "pop at the top of the next inner step" (leaf bit set as well)
struct WarpStack {
  uint32_t base;   // shared address of this thread's entry 0
  uint32_t limit;  // base + kPsStack * kPsStride: first address that lives in the spill area
  uint2** spillBase;  // in shared memory: the spill area's base pointer (only the rare path reads it)
  __device__ __forceinline__ void init(uint2* shStack, uint2** shSpill, uint2* spill, int shEntries) {
    base = uint32_t(__cvta_generic_to_shared(shStack + threadIdx.x));  // rarely needed: may be recomputed
    const uint32_t l = base + uint32_t(shEntries) * kPsStride;
    asm volatile("mov.u32 %0, %1;" : "=r"(limit) : "r"(l));  // opaque: compared at every push / pop, kept in a register
    if (threadIdx.x == 0) *shSpill = spill;
    __syncthreads();
    spillBase = shSpill;
  }
  // rare path (trees deeper than kShStack): everything is derived here so nothing of it stays live
  __device__ __noinline__ static uint2* spillSlot(uint2** spillBase, uint32_t off) {
    return *spillBase + size_t(blockIdx.x * kTraceBlock + threadIdx.x) * kSpillEntries + off / kPsStride;
  }
  __device__ __forceinline__ void put(uint32_t sa, uint32_t ref, float d) const {
    asm volatile("st.shared.v2.u32 [%0], {%1, %2};" ::"r"(sa), "r"(ref), "r"(__float_as_uint(d)));
  }
  // push / pop under a lane predicate: the shared-memory access is a single predicated instruction and
  // only the (rare) spill case branches.
  __device__ __forceinline__ void pushIf(bool on, uint32_t& sa, uint32_t ref, float d) const {
    if (on && sa < limit) put(sa, ref, d);
    if (on && sa >= limit) {
      if (sa < base + uint32_t(kMaxStack + 1) * kPsStride) *spillSlot(spillBase, sa - limit) = make_uint2(ref, __float_as_uint(d));
    }
    if (on) sa += kPsStride;
  }
  __device__ __forceinline__ void popIf(bool on, uint32_t& sa, uint32_t& ref, float& d) const {
    if (on) sa -= kPsStride;
    uint32_t x = ref, y = __float_as_uint(d);
    if (on && sa < limit) asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(x), "=r"(y) : "r"(sa));
    if (on && sa >= limit) {
      const uint2 v = *spillSlot(spillBase, sa - limit);
      x = v.x, y = v.y;
    }
    ref = x;
    d = __uint_as_float(y);
  }
  __device__ __forceinline__ void pop(uint32_t& sa, uint32_t& ref, float& d) const { popIf(true, sa, ref, d); }
};

// One 64-byte inner-node record as two 256-bit read-only loads (LDG.E.256, new on sm_100): half the
// L1 wavefronts of four 128-bit loads — the traversal kernels are bound by the LSU data pipe.
struct NodeRec {
  float f[16];
};
__device__ __forceinline__ NodeRec loadNode(const float4* p) {
  NodeRec n;
  asm volatile("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=f"(n.f[0]), "=f"(n.f[1]), "=f"(n.f[2]), "=f"(n.f[3]), "=f"(n.f[4]), "=f"(n.f[5]), "=f"(n.f[6]), "=f"(n.f[7])
               : "l"(p));
  asm volatile("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=f"(n.f[8]), "=f"(n.f[9]), "=f"(n.f[10]), "=f"(n.f[11]), "=f"(n.f[12]), "=f"(n.f[13]), "=f"(n.f[14]), "=f"(n.f[15])
               : "l"(p + 2));
  return n;
}
#endif

// What a NEE (any-hit) ray accumulates: Hit::attenuation (hit.hpp:12).
struct TraceState {
  HitRec hit;
  V3 attenuation;
};

// testTriangle + the per-leaf loop of testBVH.  Returns true if this triangle was accepted.
template <bool NEE, bool ALPHA, bool COUNT>
YB_DEV bool testTriangle(const DScene& sc, const YcMesh& mesh, const LocalRay& r, const float4 a, const float4 b,
                         const float4 c, int nodeIdx, TraceState& st, Sampler* smp, TraceCounters& cnt) {
  if (COUNT) cnt.tri++;
  const V3 p0(a.x, a.y, a.z), p1(a.w, b.x, b.y), p2(b.z, b.w, c.x);
  const uint32_t prim = __float_as_uint(c.y), flags = __float_as_uint(c.z);
  const V3 edge1 = p1 - p0;
  const V3 edge2 = p2 - p0;
  const V3 rayEdge2 = cross(r.d, edge2);
  const float det = dot(edge1, rayEdge2);
  const bool backSide = det < 0;
  if (double(fabsf(det)) < 1e-12) return false;  // epsilon is a double, math_base.hpp:11
  const float invDet = 1.0f / det;
  const V3 bb = r.o - p0;
  const float u = dot(bb, rayEdge2) * invDet;
  if (u < 0.0f || u > 1.0f) return false;
  const V3 bEdge1 = cross(bb, edge1);
  const float v = dot(r.d, bEdge1) * invDet;
  if (v < 0.0f || u + v > 1.0f) return false;
  const float t = dot(edge2, bEdge1) * invDet;
  if (t <= kTMin || st.hit.t <= t) return false;

  if ((ALPHA && (flags & YC_TRI_ALPHA)) || (NEE && (flags & YC_TRI_TRANSPARENT))) {
    // slow path: needs interpolated uv / normal and the material
    const uint32_t gp = mesh.primOffset + prim;
    const uint32_t i0 = sc.primIndices[3 * size_t(gp)] + mesh.vertOffset,
                   i1 = sc.primIndices[3 * size_t(gp) + 1] + mesh.vertOffset,
                   i2 = sc.primIndices[3 * size_t(gp) + 2] + mesh.vertOffset;
    const YcMaterial& mat = sc.materials[sc.primMaterial[gp]];
    const float w = 1.0f - u - v;
    const V2 uv0(sc.uvs[2 * size_t(i0)], sc.uvs[2 * size_t(i0) + 1]), uv1(sc.uvs[2 * size_t(i1)], sc.uvs[2 * size_t(i1) + 1]),
      uv2(sc.uvs[2 * size_t(i2)], sc.uvs[2 * size_t(i2) + 1]);
    const V2 uv = w * uv0 + u * uv1 + v * uv2;
    if (ALPHA && (flags & YC_TRI_ALPHA)) {
      float alpha = materialAlpha(sc, mat, uv);
      if (alpha < 1.0f && smp->get1D() > alpha) return false;  // draw only when alpha < 1 (short-circuit)
    }
    if (NEE && (flags & YC_TRI_TRANSPARENT)) {
      const V3 n = w * V3(sc.normals + 3 * size_t(i0)) + u * V3(sc.normals + 3 * size_t(i1)) +
                   v * V3(sc.normals + 3 * size_t(i2));
      st.attenuation *= absDot(n, r.d) * materialBase(sc, mat, uv);
      return false;
    }
  }
  st.hit.t = t;
  st.hit.u = u;
  st.hit.v = v;
  st.hit.prim = prim;
  st.hit.node = nodeIdx;
  st.hit.backSide = backSide ? 1u : 0u;
  return true;
}

// testBVH for one mesh.  EARLY_OUT (NEE only, scenes without alpha-tested materials): stop at the
// first accepted occluder — the reference keeps walking, but an occluded NEE sample is discarded
// whatever else it would have found (mis-integrator.cpp:121), so the image is identical.
template <bool NEE, bool ALPHA, bool COUNT, bool EARLY_OUT>
YB_DEV bool testBVH(const DScene& sc, const YcMesh& mesh, const LocalRay& r, int nodeIdx, TraceState& st,
                    TravStack& stack, Sampler* smp, TraceCounters& cnt) {
  float d;
  if (!slab<COUNT>(r, V3(mesh.rootMin), V3(mesh.rootMax), kTMin, st.hit.t, d, cnt)) return false;
  const float4* __restrict__ nodes = sc.bvhNodes + 4 * size_t(mesh.nodeOffset);
  const float4* __restrict__ tris = sc.bvhTris + 3 * size_t(mesh.triOffset);
  uint32_t cur = mesh.rootRef;
  int sp = 0;
  bool didHit = false;
  while (true) {
    if (d < st.hit.t) {
      if (cur & YC_REF_LEAF) {
        uint32_t ti = cur & ~YC_REF_LEAF;
        while (true) {
          const float4 a = __ldg(tris + 3 * size_t(ti)), b = __ldg(tris + 3 * size_t(ti) + 1),
                       c = __ldg(tris + 3 * size_t(ti) + 2);
          didHit |= testTriangle<NEE, ALPHA, COUNT>(sc, mesh, r, a, b, c, nodeIdx, st, smp, cnt);
          if (NEE && didHit) break;  // ray-integrator.cpp:121: leaves the leaf loop only
          if (__float_as_uint(c.z) & YC_TRI_LAST) break;
          ti++;
        }
        if (NEE && EARLY_OUT && didHit) return true;
        if (sp == 0) break;
        stack.pop(--sp, cur, d);
      } else {
        const float4 n0 = __ldg(nodes + 4 * size_t(cur)), n1 = __ldg(nodes + 4 * size_t(cur) + 1),
                     n2 = __ldg(nodes + 4 * size_t(cur) + 2), n3 = __ldg(nodes + 4 * size_t(cur) + 3);
        float d1, d2;
        bool hit1 = slab<COUNT>(r, V3(n0.x, n0.y, n0.z), V3(n0.w, n1.x, n1.y), kTMin, st.hit.t, d1, cnt);
        bool hit2 = slab<COUNT>(r, V3(n1.z, n1.w, n2.x), V3(n2.y, n2.z, n2.w), kTMin, st.hit.t, d2, cnt);
        uint32_t c1 = __float_as_uint(n3.x), c2 = __float_as_uint(n3.y);
        if (hit1) {
          if (hit2) {
            if (d1 > d2) {
              float td = d1; d1 = d2; d2 = td;
              uint32_t tc = c1; c1 = c2; c2 = tc;
            }
            stack.push(sp++, c2, d2);
          }
          cur = c1;
          d = d1;
        } else if (hit2) {
          cur = c2;
          d = d2;
        } else {
          if (sp == 0) break;
          stack.pop(--sp, cur, d);
        }
      }
    } else {
      if (sp == 0) break;
      stack.pop(--sp, cur, d);
    }
  }
  return didHit;
}

// A BVH layout as the scene walks use it: what differs between the reference-order BVH2 (here) and the 4-wide
// quantised BVH (WideWalk, wide_bvh.cuh).
//   Ray               per-ray box state, set(o, d); a LocalRay whose o / d the triangle tests read
//   box<COUNT>        float-corner box test (scene-graph node boxes, mesh root boxes)
//   mesh<…>           one mesh's sequential walk (traceScene)
// and, for the persistent kernels only (CUDA):
//   nodes, rootRef    mesh mi's node array and root ref
//   parks(COUNT)      whether the persistent walk parks leaves; kParkBelow: int32_t(ref) < kParkBelow is a leaf to park
//   inner<COUNT>      one inner-node visit of the persistent walk: the next `cur` / `dcur` (kPopRef: pop), pushes
struct Bvh2Walk {
  using Ray = LocalRay;
  template <bool COUNT>
  YB_DEV static bool box(const Ray& r, V3 lo, V3 hi, float tmx, float& d, TraceCounters& cnt) {
    return slab<COUNT>(r, lo, hi, kTMin, tmx, d, cnt);
  }
  template <bool NEE, bool ALPHA, bool COUNT, bool EARLY_OUT>
  YB_DEV static bool mesh(const DScene& sc, int mi, const Ray& r, int nodeIdx, TraceState& st, TravStack& stack, Sampler* smp,
                          TraceCounters& cnt) {
    return testBVH<NEE, ALPHA, COUNT, EARLY_OUT>(sc, sc.meshes[mi], r, nodeIdx, st, stack, smp, cnt);
  }
#ifndef YB_HOSTSIM
  __device__ __forceinline__ static const float4* nodes(const DScene& sc, int, const YcMesh& mesh) {
    return sc.bvhNodes + 4 * size_t(mesh.nodeOffset);
  }
  __device__ __forceinline__ static uint32_t rootRef(const DScene&, int, const YcMesh& mesh) { return mesh.rootRef; }
  // counting builds reproduce the reference's box-test counts: no parking there
  __host__ __device__ static constexpr bool parks(bool count) { return !count; }
  static constexpr int32_t kParkBelow = -2;  // a leaf (bit 31) other than kNoRef / kPopRef
  template <bool COUNT>
  __device__ __forceinline__ static void inner(const Ray& r, const float4* nodes, float hitT, const WarpStack& stack, uint32_t& sp,
                                               uint32_t& cur, float& dcur, const TraceTuning&, TraceCounters& cnt) {
    const NodeRec nr = loadNode(nodes + 4 * size_t(cur));
    // testBVH's pop-time cull `d < hit.t` (ray-integrator.cpp:100): an entry that fails it is
    // dropped without testing its children — here both tests are made to fail (tmax = -inf)
    const bool live = dcur < hitT;
    const float tmx = live ? hitT : -INFINITY;
    float d1, d2;
    const bool hit1 = slabLive(r, V3(nr.f[0], nr.f[1], nr.f[2]), V3(nr.f[3], nr.f[4], nr.f[5]), kTMin, tmx, d1);
    const bool hit2 = slabLive(r, V3(nr.f[6], nr.f[7], nr.f[8]), V3(nr.f[9], nr.f[10], nr.f[11]), kTMin, tmx, d2);
    if (COUNT && live) cnt.box += 2;
    const uint32_t c1 = __float_as_uint(nr.f[12]), c2 = __float_as_uint(nr.f[13]);
    // testBVH's descend / push / pop decisions (ray-integrator.cpp:131-152) as selects
    const bool both = hit1 && hit2;
    const bool swapped = both && d1 > d2;
    const bool first = hit1 && !swapped;
    const uint32_t farRef = swapped ? c1 : c2;
    const float farD = swapped ? d1 : d2;
    const uint32_t nearRef = first ? c1 : c2;
    const float nearD = first ? d1 : d2;
    stack.pushIf(both, sp, farRef, farD);
    cur = (hit1 || hit2) ? nearRef : kPopRef;
    dcur = nearD;
  }
#endif
};

// testNode over the whole scene graph (DFS pre-order with skip links instead of recursion), each mesh walked in
// Walk's layout.  `st.hit.t` must be preset (inf for closest hits, tMax for NEE rays).  Returns didHit.
template <class Walk, bool NEE, bool ALPHA, bool COUNT, bool EARLY_OUT>
YB_DEV bool traceScene(const DScene& sc, V3 origin, V3 dir, TraceState& st, TravStack& stack, Sampler* smp,
                       TraceCounters& cnt) {
  V3 ro[YC_MAX_NODE_DEPTH + 1], rd[YC_MAX_NODE_DEPTH + 1];
  ro[0] = origin;
  rd[0] = dir;
  bool didHit = false;
  uint32_t i = 0;
  while (i < sc.nNodes) {
    const YcNode& nd = sc.nodes[i];
    const int k = nd.depth;
    typename Walk::Ray r;
    // ray-integrator.cpp:26-30: transform.inverse(origin, Point), inverse(dir, Vector); dir NOT renormalised
    r.set(xformRows(nd.inv, ro[k], 1.0f), xformRows(nd.inv, rd[k], 0.0f));
    ro[k + 1] = r.o;
    rd[k + 1] = r.d;
    float d;
    if (!Walk::template box<COUNT>(r, V3(nd.bmin), V3(nd.bmax), st.hit.t, d, cnt) || st.hit.t < d) {
      i = uint32_t(nd.skip);
      continue;
    }
    if (nd.mesh >= 0) {
      const bool h = Walk::template mesh<NEE, ALPHA, COUNT, EARLY_OUT>(sc, nd.mesh, r, int(i), st, stack, smp, cnt);
      didHit |= h;
      if (NEE && EARLY_OUT && h) return true;
    }
    i++;
  }
  return didHit;
}

// Ray in the object space of `node`, rebuilt by walking the ancestor chain root → node
// (same sequence of transforms as the recursion in testNode).
YB_DEV void localRayAt(const DScene& sc, int node, V3 origin, V3 dir, V3& o, V3& d) {
  int chain[YC_MAX_NODE_DEPTH];
  int n = 0;
  for (int k = node; k >= 0; k = sc.nodes[k].parent) chain[n++] = k;
  o = origin;
  d = dir;
  for (int k = n - 1; k >= 0; k--) {
    const YcNode& nd = sc.nodes[chain[k]];
    V3 no = xformRows(nd.inv, o, 1.0f), ndir = xformRows(nd.inv, d, 0.0f);
    o = no;
    d = ndir;
  }
}

// Full Hit as the reference holds it after testNode returns to the caller:
// testMesh (ray-integrator.cpp:56-82) then the way back up the recursion (:50-52).
struct SurfaceHit {
  V3 p, n, tg;
  V2 uv;
  int material;
  int lightIdx;
};

YB_DEV V3 shadingNormal(const DScene& sc, const YcMaterial& mat, V3 n, V3 t, float tw, V2 uv) {
  // BSDF::normal, core/bsdf.cpp:43-58 (m_normalScale is never applied)
  if (mat.normalTex >= 0) {
    V3 sampled = sampleU8RGB(sc, mat.normalTex, uv) * 2.0f - 1.0f;
    Frame f(n, t, tw);
    return normalized(f.ltw(sampled));
  }
  return n;
}

YB_DEV SurfaceHit resolveHit(const DScene& sc, const HitRec& h, V3 origin, V3 dir) {
  SurfaceHit s;
  const YcNode& nd = sc.nodes[h.node];
  const YcMesh& mesh = sc.meshes[nd.mesh];
  V3 lo, ld;
  localRayAt(sc, h.node, origin, dir, lo, ld);
  const uint32_t gp = mesh.primOffset + h.prim;
  const size_t i0 = sc.primIndices[3 * size_t(gp)] + mesh.vertOffset, i1 = sc.primIndices[3 * size_t(gp) + 1] + mesh.vertOffset,
               i2 = sc.primIndices[3 * size_t(gp) + 2] + mesh.vertOffset;
  const float u = h.u, v = h.v;
  const float w = 1.0f - u - v;
  // testTriangle accept path (ray-integrator.cpp:205-227)
  s.uv = w * V2(sc.uvs[2 * i0], sc.uvs[2 * i0 + 1]) + u * V2(sc.uvs[2 * i1], sc.uvs[2 * i1 + 1]) +
         v * V2(sc.uvs[2 * i2], sc.uvs[2 * i2 + 1]);
  V3 n = w * V3(sc.normals + 3 * i0) + u * V3(sc.normals + 3 * i1) + v * V3(sc.normals + 3 * i2);
  s.p = lo + (h.t * ld);
  s.material = int(sc.primMaterial[gp]);
  // testMesh (ray-integrator.cpp:63-79)
  const float* t0 = sc.tangents + 4 * i0;
  const float* t1 = sc.tangents + 4 * i1;
  const float* t2 = sc.tangents + 4 * i2;
  V3 tg3 = w * V3(t0) + u * V3(t1) + v * V3(t2);
  float tgw = t0[3] * w + t1[3] * u + t2[3] * v;
  n = shadingNormal(sc, sc.materials[s.material], n, tg3, tgw, s.uv);
  const V3 axisY(0.0f, 1.0f, 0.0f);
  if (absDot(n, axisY) > 0.999f) s.tg = V3(1.0f, 0.0f, 0.0f);
  else s.tg = normalized(cross(n, axisY));
  s.lightIdx = sc.primLight[gp];
  // back up the recursion: every ancestor (including the hit node) applies its transform
  V3 p = s.p;
  for (int k = h.node; k >= 0; k = sc.nodes[k].parent) {
    const YcNode& a = sc.nodes[k];
    p = xformRows(a.fwd, p, 1.0f);           // Transform::Type::Point
    n = normalized(mul3x3(a.nrm, n));        // Type::Normal (normalised, transform.hpp:71)
    s.tg = xformRows(a.fwd, s.tg, 0.0f);     // Type::Vector
  }
  s.p = p;
  s.n = n;
  return s;
}

}  // namespace yb
