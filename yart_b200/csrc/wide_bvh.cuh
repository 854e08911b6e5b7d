// wide_bvh.cuh — the GPU-friendly wide-node layout of the reference's SAH BVH (BASELINE.json north_star:
// "flattens the same SAH BVH into a GPU-friendly wide-node layout") and its traversal.
//
// yc_upload_scene collapses every mesh's BVH2 (the reference's tree, src/core/bvh.hpp:21-33, as it arrives in
// YcScene::bvhNodes) into 4-wide nodes with QUANTISED child boxes (after Ylitie, Karras, Laine, "Efficient
// incoherent ray traversal on GPUs through compressed wide BVHs", HPG 2017 — here 4-wide with explicit child refs):
// same leaves (the same contiguous triangle runs of YcScene::bvhTris, so the triangle arithmetic and every
// accepted hit's t / u / v are the reference's), inner levels removed greedily by surface area.
//
//   WideNode, 64 B = 2 x LDG.256 (the uncompressed 128-B version of this node — 7 x LDG.128 per visit — ran at 95 %
//   of the L1's tag-stage throughput and was slower than the BVH2 walk: profiles/README.md, round 2):
//       S.x S.y S.z            2^15 quanta per axis; the quantum Q = 2^e is the smallest with 255 * Q >= extent    12 B
//       p'.x p'.y p'.z         grid origin P (at or below the node's low corner) minus S, rounded down            12 B
//       qlo.x qhi.x qlo.y qhi.y qlo.z qhi.z   one byte per child: plane = P + q * Q, rounded OUTWARDS            24 B
//                              (floor / ceil with a 1/128-quantum guard), so a quantised box contains the child's box
//       ref[4]                 YcBvhNode::ref encoding, kWideEmpty = unused slot                                   16 B
//   Per visit a lane forms, per axis,  Sd = S / d  and  Bn, Bf = (p' - o) / d  moved down / up by the origin term below
//   (one FMUL + three FFMA), and per child plane one PRMT that drops the byte into mantissa bits 8..15 of 1.0f
//   (v = 1 + q / 32768, exact) and one FFMA  t = v * Sd + B = (P + q * Q - o) / d;  near / far planes are picked per
//   axis on the packed words with the ray's sign masks (6 bit-selects per visit, not 24).
//
// Error bound of the box test (u = 2^-24; per axis, w = 1 / d exactly, X = a plane, o the ray origin; every float
// operation rounds to nearest, so each contributes a relative error of at most u):
//   idir = w (1 + e1),  odir = -o idir (1 + e2),  Sd = S idir (1 + e3),  Bd = (p' idir + odir) (1 + e4),
//   t = (v Sd + Bd) (1 + e5).  With X = p' + v S exactly this is
//     t = (1 + e1)(1 + e5) [ (X - o) w  +  v S w e3  +  (p' - o) w e4  -  o w e2 (1 + e4) ],
//   and since |p' - o| <= |X - o| + v S:
//     |t - (X - o) w|  <=  2.02 u v S |w|  +  3 u |X| |w|  +  4 u |o| |w|   (to first order in u).
//   * 2.02 u v S |w| <= Q |w| / 253 (v < 1.008, S = 2^15 Q): held by the 1/128-quantum guard of the outward rounding.
//   * the |X| term is held by growing every child box by kWideSlack |corner| before quantising (host, exact in double;
//     float-corner boxes in slabWideBox: at run time).
//   * the |o| term is held per ray: odn = odir - kWideSlack |odir| feeds the near planes, odir + >= kWideSlack |odir|
//     (farOffset) the far ones; that fused add is one more rounding inside B, covered by the same terms.
// kWideSlack = 16 u also covers what testTriangle's own float arithmetic does to an accepted hit: s = o - p0 and its
// cross and dot products round relative to each component of s, which moves the tested ray by up to ~6 u |o - p0| per
// axis, that is 6 u (|o| + |X|) |w| in t.  So the computed [near, far] of a box contains the t of every hit that
// testTriangle accepts inside it (tests/test_wide_bvh_robustness.py checks this against a float64 brute force at far
// origins and tiny nodes), except where det is so small that the triangle test's t itself is off by more than the
// slack (rays grazing a triangle's plane: relative t error ~ u / sin of the angle).  Planes whose S would not be a
// finite float (extents beyond ~1.3e36) or non-finite boxes are refused: the scene then has no wide layout.
//
// What differs from the reference-order BVH2 walk (traverse.cuh), and why results still match:
//   * box culling only.  The set of triangles tested is a superset / reordering of the reference's (bound above), every
//     triangle test is the reference's arithmetic (testTriangle, -fmad=false), and the closest hit is the
//     minimum over accepted tests.  Hit ids / t / u / v are therefore identical except where two triangles tie
//     in t to the last bit, or where a hit sits on the boundary of a box that the reference's own slab test
//     (`bmin * idir + odir`, two roundings, not conservative) culls: there the wide walk finds the hit and the
//     reference misses it.  tests/ count those.
//   * a zero direction component is clamped to ±1e-20 for the BOX test only (Aila-Laine), so a ray with
//     d.x == 0 and o.x == 0 no longer has NaN slabs on that axis and no longer walks every box that overlaps
//     it in y and z (14 K boxes for one ray of the C2 camera, profiles/README.md "Pathological rays").
//   * used only for scenes without alpha-tested materials: there the order of triangle tests cannot move a
//     sampler draw (ray-integrator.cpp:211).  Alpha scenes keep the reference-order BVH2 walk.
//   * NEE rays through thin transmissive surfaces multiply Hit::attenuation in a different order
//     (floating-point product order; last-bit differences in those pixels).
#pragma once
#include <vector>

#include "traverse.cuh"

#include <atomic>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <thread>

namespace yb {

constexpr uint32_t kWideEmpty = 0xfffffffdu;  // unused child slot (has the leaf bit; never equals a real leaf ref)
constexpr float kWideSlack = 0x1p-20f;  // 16 float ulps of 1: the relative widening of the bound in the header
constexpr int kWideMaxExp = 112;        // largest quantum exponent: S = 2^(e + 15) stays a finite float

struct WideNode {
  float pS[3];      // p' = P - S per axis (rounded down)
  float S[3];       // 2^(e + 15)
  uint32_t q[6];    // qlo.x, qhi.x, qlo.y, qhi.y, qlo.z, qhi.z; byte k = child k
  uint32_t ref[4];
};
static_assert(sizeof(WideNode) == 64, "WideNode is two 32-byte sectors");

// ---- host: BVH2 → BVH4 collapse --------------------------------------------------------------------
// Appends mesh `m`'s wide nodes to `out` (children of a node are allocated together, parents before children)
// and returns the deepest level (root = 1; 0 for a single-leaf mesh).
// Two passes: the walk that decides which BVH2 nodes open into which wide node (sequential: a node's children are
// numbered when it is visited) and the quantisation of every wide node's child boxes (independent per node, double
// arithmetic: spread over the host's cores).
struct WideChildBox {
  float lo[3], hi[3];
  uint32_t ref;  // BVH2 ref while collapsing, then the wide ref
};
struct WideDraft {
  WideChildBox c[4];
  int n;
};
// Quantises one wide node's child boxes; false when an axis cannot be put on a grid with a finite float S and p'
// (extents beyond ~1.3e36, or non-finite boxes): the scene then has no wide layout.
inline bool quantiseWideNode(const WideDraft& d, WideNode& node) {
  const WideChildBox* c = d.c;
  const int n = d.n;
  node = WideNode{};
  // Quantisation grid per axis: quantum Q = 2^e, S = 2^15 Q, p' = the float at or below (low corner - S), grid
  // origin P = p' + S (<= the low corner; P, q * Q and their sums are exact in double).  e is the smallest exponent
  // for which the planes fit in a byte with the guard below.  The boxes quantised are the children's boxes grown by
  // kWideSlack of their corners' magnitudes (the position term of the bound in the header).
  for (int a = 0; a < 3; a++) {
    double cl[4], ch[4];
    double lo = INFINITY, hi = -INFINITY;
    for (int k = 0; k < n; k++) {
      cl[k] = double(c[k].lo[a]) - double(kWideSlack) * std::fabs(double(c[k].lo[a]));
      ch[k] = double(c[k].hi[a]) + double(kWideSlack) * std::fabs(double(c[k].hi[a]));
      lo = std::min(lo, cl[k]), hi = std::max(hi, ch[k]);
    }
    if (!std::isfinite(lo) || !std::isfinite(hi)) return false;
    int e = -100;
    if (hi - lo > 0.0) std::frexp((hi - lo) / 254.0, &e);
    e = std::max(-100, e);
    for (;; e++) {
      if (e > kWideMaxExp) return false;
      const double Q = std::ldexp(1.0, e), S = std::ldexp(1.0, e + 15);
      float pS = float(lo - S - Q / 64);  // the origin sits 1/64 quantum below the low corner: a guard for q = 0 too
      if (double(pS) > lo - S - Q / 64) pS = std::nextafterf(pS, -INFINITY);
      if (!std::isfinite(pS)) return false;
      const double P = double(pS) + S;
      // outward rounding with a 1/128-quantum guard: it holds the S-proportional rounding of the device's plane
      // distances (header: at most Q / 253)
      bool fits = true;
      uint32_t ql[4], qh[4];
      for (int k = 0; k < n && fits; k++) {
        const double l = std::floor((cl[k] - P) / Q - 1.0 / 128), h = std::ceil((ch[k] - P) / Q + 1.0 / 128);
        fits = l >= 0.0 && h <= 255.0;
        ql[k] = uint32_t(std::max(0.0, l)), qh[k] = uint32_t(std::max(0.0, std::min(255.0, h)));
      }
      if (!fits) continue;
      node.pS[a] = pS, node.S[a] = float(S);
      for (int k = 0; k < 4; k++) {
        // unused slots: lo = 255, hi = 0 — an empty interval on every axis
        node.q[2 * a] |= (k < n ? ql[k] : 255u) << (8 * k);
        node.q[2 * a + 1] |= (k < n ? qh[k] : 0u) << (8 * k);
      }
      break;
    }
  }
  for (int k = 0; k < 4; k++) node.ref[k] = k < n ? c[k].ref : kWideEmpty;
  return true;
}

// One step of the collapse: the wide node that the BVH2 inner node `ref2` opens into (greedy by surface area, the
// reference tree's left-to-right order kept).  Children that are BVH2 inner nodes keep their BVH2 ref in `d.c[k].ref`.
inline void openWideNode(const YcBvhNode* bvh2, uint32_t ref2, WideDraft& d) {
  WideChildBox* c = d.c;
  int n = 0;
  auto put = [&](WideChildBox& dst, const float* lo, const float* hi, uint32_t ref) {
    memcpy(dst.lo, lo, 12), memcpy(dst.hi, hi, 12), dst.ref = ref;
  };
  auto area = [](const WideChildBox& b) {
    const float dx = b.hi[0] - b.lo[0], dy = b.hi[1] - b.lo[1], dz = b.hi[2] - b.lo[2];
    return dx * dy + dy * dz + dz * dx;
  };
  {
    const YcBvhNode& nd = bvh2[ref2];
    put(c[0], nd.c0min, nd.c0max, nd.ref0), put(c[1], nd.c1min, nd.c1max, nd.ref1);
    n = 2;
  }
  while (n < 4) {
    int best = -1;
    float bestArea = -1.0f;
    for (int k = 0; k < n; k++)
      if (!(c[k].ref & YC_REF_LEAF) && area(c[k]) > bestArea) best = k, bestArea = area(c[k]);
    if (best < 0) break;
    // the opened child's slot receives its left child, its right child is inserted after it
    const YcBvhNode& nd = bvh2[c[best].ref];
    for (int k = n - 1; k > best; k--) c[k + 1] = c[k];
    put(c[best], nd.c0min, nd.c0max, nd.ref0), put(c[best + 1], nd.c1min, nd.c1max, nd.ref1);
    n++;
  }
  d.n = n;
}

// Collapses the subtree under BVH2 node `ref2` into `drafts` (index 0 = the subtree's root; children are numbered when
// their parent is visited).  `limit` > 0: stop opening once that many subtrees are pending and report them in
// `pending` as (BVH2 ref, draft index) — the caller finishes those elsewhere.  Returns the deepest level reached.
struct WidePending {
  uint32_t ref2, draft;
  int depth;
};
inline int collapseSubtree(const YcBvhNode* bvh2, uint32_t ref2, int depth0, std::vector<WideDraft>& drafts, size_t limit,
                           std::vector<WidePending>* pending) {
  drafts.assign(1, WideDraft{});
  std::vector<WidePending> todo{{ref2, 0u, depth0}};
  int maxDepth = depth0;
  size_t head = 0;  // breadth-first while a limit is set (an even split of the work), depth-first otherwise
  while (head < todo.size()) {
    if (limit && todo.size() - head >= limit) break;
    WidePending w;
    if (limit) {
      w = todo[head++];
    } else {
      w = todo.back();
      todo.pop_back();
    }
    maxDepth = std::max(maxDepth, w.depth);
    WideDraft d;
    openWideNode(bvh2, w.ref2, d);
    for (int k = 0; k < d.n; k++) {
      if (d.c[k].ref & YC_REF_LEAF) continue;
      const uint32_t wide = uint32_t(drafts.size());
      __builtin_prefetch(&bvh2[d.c[k].ref]);
      todo.push_back({d.c[k].ref, wide, w.depth + 1});
      d.c[k].ref = wide;
      drafts.emplace_back();
    }
    drafts[w.draft] = d;
  }
  if (pending) pending->assign(todo.begin() + long(head), todo.end());
  return maxDepth;
}

// Returns the deepest level, or -1 when a node's boxes cannot be quantised (quantiseWideNode).
inline int collapseToWide(const YcBvhNode* bvh2, const YcMesh& m, std::vector<WideNode>& out, WideMesh& wm) {
  wm.nodeOffset = uint32_t(out.size());
  wm.rootRef = m.rootRef;
  if (m.rootRef & YC_REF_LEAF) return 0;
  const char* traceEnv = getenv("YART_B200_BUILD_TRACE");
  const bool trace = traceEnv && *traceEnv && *traceEnv != '0';
  const auto tw = std::chrono::high_resolution_clock::now();
  unsigned threads = std::max(1u, std::min(16u, std::thread::hardware_concurrency()));
  if (m.nInner < 50000) threads = 1;
  // the top of the tree on this thread until there are enough pending subtrees to share out, then one subtree at a
  // time per worker into its own array; the pieces are appended and their references shifted afterwards
  std::vector<WideDraft> top;
  std::vector<WidePending> pending;
  int maxDepth = collapseSubtree(bvh2, m.rootRef, 1, top, threads > 1 ? size_t(threads) * 8 : 0, &pending);
  std::vector<std::vector<WideDraft>> parts(pending.size());
  std::vector<int> depths(pending.size(), 0);
  if (!pending.empty()) {
    std::atomic<size_t> next{0};
    auto work = [&] {
      for (size_t i; (i = next.fetch_add(1)) < pending.size();)
        depths[i] = collapseSubtree(bvh2, pending[i].ref2, pending[i].depth, parts[i], 0, nullptr);
    };
    std::vector<std::thread> pool;
    for (unsigned t = 0; t < threads; t++) pool.emplace_back(work);
    for (auto& th : pool) th.join();
  }
  // layout: the top's drafts first (the pending subtrees' roots already have their slots there), then every part
  // without its root
  std::vector<size_t> partBase(parts.size());
  size_t count = top.size();
  for (size_t i = 0; i < parts.size(); i++) {
    partBase[i] = count;
    count += parts[i].size() - 1;
    maxDepth = std::max(maxDepth, depths[i]);
  }
  const auto tq = std::chrono::high_resolution_clock::now();
  const size_t base = out.size();
  out.resize(base + count);
  std::atomic<bool> quantised{true};
  auto emitTop = [&](size_t lo, size_t hi) {
    for (size_t i = lo; i < hi; i++)
      if (!quantiseWideNode(top[i], out[base + i])) quantised = false;
  };
  auto emitPart = [&](size_t p) {
    // local index 0 is the part's root, which lives in the top's slot; local index j >= 1 lives at partBase + j - 1
    std::vector<WideDraft>& part = parts[p];
    for (size_t j = 0; j < part.size(); j++) {
      WideDraft d = part[j];
      for (int k = 0; k < d.n; k++)
        if (!(d.c[k].ref & YC_REF_LEAF)) d.c[k].ref = uint32_t(partBase[p] + d.c[k].ref - 1);
      if (!quantiseWideNode(d, out[base + (j == 0 ? size_t(pending[p].draft) : partBase[p] + j - 1)])) quantised = false;
    }
  };
  if (threads == 1) {
    emitTop(0, top.size());
    for (size_t p = 0; p < parts.size(); p++) emitPart(p);
  } else {
    // the pending roots' slots in `top` are placeholders: their real content comes from the parts
    std::vector<char> isPendingRoot(top.size(), 0);
    for (const WidePending& w : pending) isPendingRoot[w.draft] = 1;
    std::atomic<size_t> next{0};
    auto work = [&] {
      for (size_t i; (i = next.fetch_add(1)) < parts.size() + 1;) {
        if (i == parts.size()) {
          for (size_t t = 0; t < top.size(); t++)
            if (!isPendingRoot[t] && !quantiseWideNode(top[t], out[base + t])) quantised = false;
        } else {
          emitPart(i);
        }
      }
    };
    std::vector<std::thread> pool;
    for (unsigned t = 0; t < threads; t++) pool.emplace_back(work);
    for (auto& th : pool) th.join();
  }
  if (trace && count > 10000)
    fprintf(stderr, "yart_b200 wide collapse: %zu nodes, walk %.1f ms, quantisation %.1f ms\n", count,
            std::chrono::duration<double, std::milli>(tq - tw).count(),
            std::chrono::duration<double, std::milli>(std::chrono::high_resolution_clock::now() - tq).count());
  return quantised ? maxDepth : -1;
}

// ---- device ------------------------------------------------------------------------------------------
// Per-ray constants of the wide slab test.
struct WideRay {
  V3 idir;                // 1 / d (zero components clamped to ±1e-20)
  V3 odn;                 // -o * idir moved down by kWideSlack |o * idir| (near planes; farOffset: far planes)
  uint32_t mx, my, mz;    // all ones where d < 0 on that axis (the near plane of a box is its hi plane), else 0
  YB_DEV void set(V3 o, V3 d) {
    const float eps = 1e-20f;
    const float dx = fabsf(d.x) > eps ? d.x : copysignf(eps, d.x), dy = fabsf(d.y) > eps ? d.y : copysignf(eps, d.y),
                dz = fabsf(d.z) > eps ? d.z : copysignf(eps, d.z);
    idir = V3(1.0f / dx, 1.0f / dy, 1.0f / dz);
    const V3 odir(-o.x * idir.x, -o.y * idir.y, -o.z * idir.z);
    odn = V3(fmaf(fabsf(odir.x), -kWideSlack, odir.x), fmaf(fabsf(odir.y), -kWideSlack, odir.y), fmaf(fabsf(odir.z), -kWideSlack, odir.z));
    mx = dx < 0.0f ? 0xffffffffu : 0u, my = dy < 0.0f ? 0xffffffffu : 0u, mz = dz < 0.0f ? 0xffffffffu : 0u;
  }
};

// -o * idir moved up by at least kWideSlack |o * idir|, formed from odn where it is needed (one FFMA per axis, no
// register held for the whole walk): 3 kWideSlack |odn| >= 2 kWideSlack |o * idir| + the two roundings.
YB_DEV float farOffset(float odn) { return fmaf(fabsf(odn), 3.0f * kWideSlack, odn); }

#ifdef YB_HOSTSIM
YB_DEV float fmaExact(float a, float b, float c) { return fmaf(a, b, c); }
#else
YB_DEV float fmaExact(float a, float b, float c) { return __fmaf_rn(a, b, c); }
#endif

// A box given by its float corners (scene-graph node boxes, mesh root boxes): entry distance in `tn`, true when the
// slab interval [max(tn, tMin), min(tf, tmx)] is not empty.  The corners move outwards by kWideSlack of their
// magnitude first (the position term of the header's bound; quantised child planes carry it from the host).
// fmaxf / fminf drop NaN operands, like the reference's NaN-tolerant rmin / rmax.
YB_DEV bool slabWideBox(const WideRay& w, V3 lo, V3 hi, float tmn, float tmx, float& tn) {
  lo = V3(fmaf(fabsf(lo.x), -kWideSlack, lo.x), fmaf(fabsf(lo.y), -kWideSlack, lo.y), fmaf(fabsf(lo.z), -kWideSlack, lo.z));
  hi = V3(fmaf(fabsf(hi.x), kWideSlack, hi.x), fmaf(fabsf(hi.y), kWideSlack, hi.y), fmaf(fabsf(hi.z), kWideSlack, hi.z));
  const V3 nearP(w.mx ? hi.x : lo.x, w.my ? hi.y : lo.y, w.mz ? hi.z : lo.z);
  const V3 farP(w.mx ? lo.x : hi.x, w.my ? lo.y : hi.y, w.mz ? lo.z : hi.z);
  const float tnx = fmaExact(nearP.x, w.idir.x, w.odn.x), tny = fmaExact(nearP.y, w.idir.y, w.odn.y),
              tnz = fmaExact(nearP.z, w.idir.z, w.odn.z);
  const float tfx = fmaExact(farP.x, w.idir.x, farOffset(w.odn.x)), tfy = fmaExact(farP.y, w.idir.y, farOffset(w.odn.y)),
              tfz = fmaExact(farP.z, w.idir.z, farOffset(w.odn.z));
  tn = fmaxf(fmaxf(tnx, tny), fmaxf(tnz, tmn));
  const float tf = fminf(fminf(tfx, tfy), fminf(tfz, tmx));
  return tn <= tf;
}

// Byte K of `word` as v = 1 + q / 32768: the byte dropped into mantissa bits 8..15 of 1.0f (one PRMT; `one` holds the
// bits of 1.0f in a register so that the selector can be the instruction's immediate).
template <int K>
YB_DEV float planeUnit(uint32_t word, uint32_t one) {
#ifdef YB_HOSTSIM
  return __uint_as_float(__byte_perm(word, one, 0x7604u | (uint32_t(K) << 4)));
#else
  uint32_t r;
  asm("prmt.b32 %0, %1, %2, %3;" : "=r"(r) : "r"(word), "r"(one), "n"(0x7604 | (K << 4)));
  return __uint_as_float(r);
#endif
}

// The four quantised child boxes of one WideNode against the ray: entry distances and hit flags (`live` false: none).
struct WideSlabs {
  float tn[4];
  bool hit[4];
};
template <int K>
YB_DEV void slabWideChild(WideSlabs& r, uint32_t one, uint32_t nx, uint32_t ny, uint32_t nz, uint32_t fx, uint32_t fy, uint32_t fz,
                          float Sx, float Sy, float Sz, float Bnx, float Bny, float Bnz, float Bfx, float Bfy, float Bfz, float tmn,
                          float tmx, bool live) {
  const float tnx = fmaExact(planeUnit<K>(nx, one), Sx, Bnx), tny = fmaExact(planeUnit<K>(ny, one), Sy, Bny),
              tnz = fmaExact(planeUnit<K>(nz, one), Sz, Bnz);
  const float tfx = fmaExact(planeUnit<K>(fx, one), Sx, Bfx), tfy = fmaExact(planeUnit<K>(fy, one), Sy, Bfy),
              tfz = fmaExact(planeUnit<K>(fz, one), Sz, Bfz);
  r.tn[K] = fmaxf(fmaxf(tnx, tny), fmaxf(tnz, tmn));
  const float tf = fminf(fminf(tfx, tfy), fminf(tfz, tmx));
  r.hit[K] = live && r.tn[K] <= tf;
}
// words: {p'.x, p'.y, p'.z, S.x, S.y, S.z, qlo.x, qhi.x} and {qlo.y, qhi.y, qlo.z, qhi.z}
YB_DEV WideSlabs slabWide4(const WideRay& w, uint32_t one, float px, float py, float pz, float sx, float sy, float sz, uint32_t qlx,
                           uint32_t qhx, uint32_t qly, uint32_t qhy, uint32_t qlz, uint32_t qhz, float tmn, float tmx, bool live) {
  const float Sx = sx * w.idir.x, Sy = sy * w.idir.y, Sz = sz * w.idir.z;
  const float Bnx = fmaExact(px, w.idir.x, w.odn.x), Bny = fmaExact(py, w.idir.y, w.odn.y), Bnz = fmaExact(pz, w.idir.z, w.odn.z);
  const float Bfx = fmaExact(px, w.idir.x, farOffset(w.odn.x)), Bfy = fmaExact(py, w.idir.y, farOffset(w.odn.y)),
              Bfz = fmaExact(pz, w.idir.z, farOffset(w.odn.z));
  // bit-select: the hi word where the ray runs against the axis
  const uint32_t nx = (qlx & ~w.mx) | (qhx & w.mx), fx = (qhx & ~w.mx) | (qlx & w.mx);
  const uint32_t ny = (qly & ~w.my) | (qhy & w.my), fy = (qhy & ~w.my) | (qly & w.my);
  const uint32_t nz = (qlz & ~w.mz) | (qhz & w.mz), fz = (qhz & ~w.mz) | (qlz & w.mz);
  WideSlabs r;
  slabWideChild<0>(r, one, nx, ny, nz, fx, fy, fz, Sx, Sy, Sz, Bnx, Bny, Bnz, Bfx, Bfy, Bfz, tmn, tmx, live);
  slabWideChild<1>(r, one, nx, ny, nz, fx, fy, fz, Sx, Sy, Sz, Bnx, Bny, Bnz, Bfx, Bfy, Bfz, tmn, tmx, live);
  slabWideChild<2>(r, one, nx, ny, nz, fx, fy, fz, Sx, Sy, Sz, Bnx, Bny, Bnz, Bfx, Bfy, Bfz, tmn, tmx, live);
  slabWideChild<3>(r, one, nx, ny, nz, fx, fy, fz, Sx, Sy, Sz, Bnx, Bny, Bnz, Bfx, Bfy, Bfz, tmn, tmx, live);
  return r;
}

// Sequential walk of one mesh's wide BVH (per-path tail kernel, CPU build of the product sources); the
// persistent-warp kernels (WideWalk::inner below) make the same decisions: the hit child with the smallest entry
// distance first (the lowest slot among equals), the other hit children pushed in slot order with their entry
// distances, popped entries culled by `d < hit.t`.
template <bool NEE, bool COUNT, bool EARLY_OUT>
YB_DEV bool testBVHWide(const DScene& sc, const YcMesh& mesh, const WideMesh& wm, const LocalRay& r, const WideRay& w,
                        int nodeIdx, TraceState& st, TravStack& stack, TraceCounters& cnt) {
  float d;
  if (COUNT) cnt.box++;
  if (!slabWideBox(w, V3(mesh.rootMin), V3(mesh.rootMax), kTMin, st.hit.t, d)) return false;
  const float4* __restrict__ nodes = sc.wideNodes + 4 * size_t(wm.nodeOffset);
  const float4* __restrict__ tris = sc.bvhTris + 3 * size_t(mesh.triOffset);
  uint32_t cur = wm.rootRef;
  int sp = 0;
  bool didHit = false;
  while (true) {
    if (d < st.hit.t) {
      if (cur & YC_REF_LEAF) {
        uint32_t ti = cur & ~YC_REF_LEAF;
        while (true) {
          const float4 a = __ldg(tris + 3 * size_t(ti)), b = __ldg(tris + 3 * size_t(ti) + 1),
                       c = __ldg(tris + 3 * size_t(ti) + 2);
          didHit |= testTriangle<NEE, false, COUNT>(sc, mesh, r, a, b, c, nodeIdx, st, nullptr, cnt);
          if (NEE && didHit) break;
          if (__float_as_uint(c.z) & YC_TRI_LAST) break;
          ti++;
        }
        if (NEE && EARLY_OUT && didHit) return true;
        if (sp == 0) break;
        stack.pop(--sp, cur, d);
      } else {
        const float4* n = nodes + 4 * size_t(cur);
        const float4 r0 = __ldg(n), r1 = __ldg(n + 1), r2 = __ldg(n + 2), rf = __ldg(n + 3);
        const uint32_t ref[4] = {__float_as_uint(rf.x), __float_as_uint(rf.y), __float_as_uint(rf.z), __float_as_uint(rf.w)};
        WideSlabs sl = slabWide4(w, 0x3f800000u, r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, __float_as_uint(r1.z), __float_as_uint(r1.w),
                                 __float_as_uint(r2.x), __float_as_uint(r2.y), __float_as_uint(r2.z), __float_as_uint(r2.w), kTMin,
                                 st.hit.t, true);
        float* tn = sl.tn;
        bool* hit = sl.hit;
        hit[2] = hit[2] && ref[2] != kWideEmpty;
        hit[3] = hit[3] && ref[3] != kWideEmpty;
        if (COUNT) cnt.box += 2u + (ref[2] != kWideEmpty) + (ref[3] != kWideEmpty);
        int nearSlot = -1;
        for (int k = 0; k < 4; k++)
          if (hit[k] && (nearSlot < 0 || tn[k] < tn[nearSlot])) nearSlot = k;
        if (nearSlot < 0) {
          if (sp == 0) break;
          stack.pop(--sp, cur, d);
        } else {
          for (int k = 0; k < 4; k++)
            if (hit[k] && k != nearSlot) stack.push(sp++, ref[k], tn[k]);
          cur = ref[nearSlot];
          d = tn[nearSlot];
        }
      }
    } else {
      if (sp == 0) break;
      stack.pop(--sp, cur, d);
    }
  }
  return didHit;
}

#ifndef YB_HOSTSIM
struct Words8 {
  uint32_t w[8];
};
__device__ __forceinline__ Words8 loadHalfNode(const float4* p) {  // 32 bytes, one sector
  Words8 r;
  asm volatile("ld.global.nc.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(r.w[0]), "=r"(r.w[1]), "=r"(r.w[2]), "=r"(r.w[3]), "=r"(r.w[4]), "=r"(r.w[5]), "=r"(r.w[6]), "=r"(r.w[7])
               : "l"(p));
  return r;
}
#endif

// The wide layout for the scene walks (members as in Bvh2Walk, traverse.cuh).  Only for scenes without alpha-tested
// materials, so triangle tests never draw from a sampler.
struct WideWalk {
  // o and d for the triangle tests (LocalRay's idir / odir are not set: the box tests use `w`)
  struct Ray : LocalRay {
    WideRay w;
    YB_DEV void set(V3 origin, V3 dir) {
      o = origin, d = dir;
      w.set(origin, dir);
    }
  };
  template <bool COUNT>
  YB_DEV static bool box(const Ray& r, V3 lo, V3 hi, float tmx, float& d, TraceCounters& cnt) {
    if (COUNT) cnt.box++;
    return slabWideBox(r.w, lo, hi, kTMin, tmx, d);
  }
  template <bool NEE, bool ALPHA, bool COUNT, bool EARLY_OUT>
  YB_DEV static bool mesh(const DScene& sc, int mi, const Ray& r, int nodeIdx, TraceState& st, TravStack& stack, Sampler*,
                          TraceCounters& cnt) {
    static_assert(!ALPHA, "the wide walk does not reproduce the order of alpha-test sampler draws");
    return testBVHWide<NEE, COUNT, EARLY_OUT>(sc, sc.meshes[mi], sc.wideMeshes[mi], r, r.w, nodeIdx, st, stack, cnt);
  }
#ifndef YB_HOSTSIM
  __device__ __forceinline__ static const float4* nodes(const DScene& sc, int mi, const YcMesh&) {
    return sc.wideNodes + 4 * size_t(sc.wideMeshes[mi].nodeOffset);
  }
  __device__ __forceinline__ static uint32_t rootRef(const DScene& sc, int mi, const YcMesh&) { return sc.wideMeshes[mi].rootRef; }
  __host__ __device__ static constexpr bool parks(bool) { return true; }
  static constexpr int32_t kParkBelow = -3;  // a leaf (bit 31) other than kNoRef / kPopRef / kWideEmpty
  // One 64-byte node = 2 x LDG.256 per lane (two L1 tag look-ups per visit instead of the BVH2 walk's two per HALF as
  // much tree), four boxes decoded with 24 PRMT + 24 FFMA, 6 selects for near / far, 16 FMNMX(3) + 4 FSETP; the nearest
  // hit child is next, the other hit children are pushed with their entry distances (predicated STS.64).
  template <bool COUNT>
  __device__ __forceinline__ static void inner(const Ray& r, const float4* nodes, float hitT, const WarpStack& stack, uint32_t& sp,
                                               uint32_t& cur, float& dcur, const TraceTuning& tune, TraceCounters& cnt) {
    // bits of 1.0f in a register ptxas cannot fold (shEntries <= 25), so that planeUnit's PRMT carries its selector as the
    // immediate instead of fetching four selectors into registers on every visit
    const uint32_t one = 0x3f800000u | (uint32_t(tune.shEntries) >> 30);
    const float4* np = nodes + 4 * size_t(cur);
    const Words8 a = loadHalfNode(np), b = loadHalfNode(np + 2);  // {p', S, q.x} and {q.y, q.z, refs}
    const uint4 rf = make_uint4(b.w[4], b.w[5], b.w[6], b.w[7]);
    // pop-time cull `d < hit.t`: a dead entry hits nothing
    const bool live = dcur < hitT;
    const WideSlabs sl = slabWide4(r.w, one, __uint_as_float(a.w[0]), __uint_as_float(a.w[1]), __uint_as_float(a.w[2]),
                                   __uint_as_float(a.w[3]), __uint_as_float(a.w[4]), __uint_as_float(a.w[5]), a.w[6], a.w[7], b.w[0],
                                   b.w[1], b.w[2], b.w[3], kTMin, hitT, live);
    const float t0 = sl.tn[0], t1 = sl.tn[1], t2 = sl.tn[2], t3 = sl.tn[3];
    const bool h0 = sl.hit[0], h1 = sl.hit[1], h2 = sl.hit[2] && rf.z != kWideEmpty, h3 = sl.hit[3] && rf.w != kWideEmpty;
    if (COUNT && live) cnt.box += 2u + (rf.z != kWideEmpty) + (rf.w != kWideEmpty);
    // nearest hit child (lowest slot among equal entry distances) → next node; the others are pushed in slot order
    const float a0 = h0 ? t0 : INFINITY, a1 = h1 ? t1 : INFINITY, a2 = h2 ? t2 : INFINITY, a3 = h3 ? t3 : INFINITY;
    const float best = fminf(fminf(a0, a1), fminf(a2, a3));
    const bool any = h0 || h1 || h2 || h3;
    const bool p0 = h0 && a0 == best, p1 = !p0 && h1 && a1 == best, p2 = !p0 && !p1 && h2 && a2 == best;
    const uint32_t nearRef = p0 ? rf.x : (p1 ? rf.y : (p2 ? rf.z : rf.w));
    const bool q0 = h0 && !p0, q1 = h1 && !p1, q2 = h2 && !p2, q3 = h3 && (p0 || p1 || p2);
    if (sp + 3u * kPsStride < stack.limit) {  // the (at most three) pushes fit in shared memory
      uint32_t sa = sp;
      if (q0) stack.put(sa, rf.x, t0), sa += kPsStride;
      if (q1) stack.put(sa, rf.y, t1), sa += kPsStride;
      if (q2) stack.put(sa, rf.z, t2), sa += kPsStride;
      if (q3) stack.put(sa, rf.w, t3), sa += kPsStride;
      sp = sa;
    } else {
      stack.pushIf(q0, sp, rf.x, t0);
      stack.pushIf(q1, sp, rf.y, t1);
      stack.pushIf(q2, sp, rf.z, t2);
      stack.pushIf(q3, sp, rf.w, t3);
    }
    cur = any ? nearRef : kPopRef;
    dcur = best;
  }
#endif
};

}  // namespace yb
