// bvh_build.cuh — the reference's binned-SAH BVH built on the GPU, node for node and index for index.
//
// Restates yart's builder (reference src/core/bvh.hpp:41-67 init, :101-113 updateBounds, :121-133 getCentroidBounds,
// :140-184 subdivide, :273-347 SahBVH::getSplit) like host/bvh_build.hpp does on the host cores, as a level-synchronous
// build: every node of a level in parallel, every triangle of every node in parallel.  What makes that possible without
// changing the tree:
//   * bounds, centroid bounds and the 3 x 20 bins are min / max / count folds — order-independent, so atomics on the
//     float bit patterns (signed-min / unsigned-max trick) give the reference's values exactly (inputs are finite: the
//     caller falls back to the host builder otherwise; the sign of a zero bound cannot arise, see DESIGN.md);
//   * the cost scan over the 19 split planes is per node and sequential, as in the reference;
//   * the reference's in-place partition (`while (i <= j) { if (c < split) i++; else swap(idx[i], idx[j--]); }`) examines
//     its elements in a fixed interleaving of a FRONT stream (positions first, first+1, ...) and a BACK stream (last,
//     last-1, ...): front elements until one belongs right, then back elements until one belongs left, and so on.
//     Left elements end up at first + (number of left elements examined before them), right elements at last - (number
//     of right elements examined before them), and both counts follow from prefix counts of the classes and from the
//     positions of the k-th right element from the front / k-th left element from the back — one scan and two
//     scatters per level (ClassK, TablesK, PartitionK below).
// Nodes of at most kSmallSpan triangles are finished by one thread each with the reference's sequential code.
// The node pool is in creation order; three more passes per tree level put it into the reference's allocation order.
// In the CPU build of the product sources (YB_HOSTSIM) the same stages run as plain loops.
#pragma once
#include <limits>
#include <vector>

#include "scan.cuh"

namespace yb {
namespace bvhb {

constexpr uint32_t kBins = 20, kMaxLeaf = 20;  // nBins bvh.hpp:283, MAX_LEAF_SIZE bvh.hpp:14
constexpr uint32_t kSmallSpan = 48;            // subtrees of at most this many triangles: one thread
constexpr uint32_t kNone = 0xffffffffu;

struct GNode {
  float mn[3], mx[3];
  uint32_t first, span;
  uint32_t left;  // pool index of the left child (right = left + 1); 0 = leaf
  uint32_t slot;  // while building: the node's slot in the next level's work list, kNone if it is not an active node
};
struct Bin {
  uint32_t count;
  float mn[3], mx[3];
};
struct NodeWork {  // per active ("big") node of the level
  uint32_t node;   // pool index
  float cmn[3], cmx[3];
  uint32_t split;  // 1: partition and create children
  uint32_t axis;
  float splitPos;
  uint32_t nLeft;
};

YB_DEV bool signBit(float v) { return (__float_as_uint(v) >> 31) != 0u; }
YB_DEV void atomMinF(float* a, float v) {
#ifdef YB_HOSTSIM
  if (v < *a || (v == *a && signBit(v))) *a = v;
#else
  if (!signBit(v)) atomicMin(reinterpret_cast<int*>(a), __float_as_int(v));
  else atomicMax(reinterpret_cast<unsigned int*>(a), __float_as_uint(v));
#endif
}
YB_DEV void atomMaxF(float* a, float v) {
#ifdef YB_HOSTSIM
  if (v > *a || (v == *a && !signBit(v))) *a = v;
#else
  if (!signBit(v)) atomicMax(reinterpret_cast<int*>(a), __float_as_int(v));
  else atomicMin(reinterpret_cast<unsigned int*>(a), __float_as_uint(v));
#endif
}
YB_DEV uint32_t atomAddU(uint32_t* a, uint32_t v) {
#ifdef YB_HOSTSIM
  const uint32_t o = *a;
  *a += v;
  return o;
#else
  return atomicAdd(a, v);
#endif
}

YB_DEV void atomMaxU(uint32_t* a, uint32_t v) {
#ifdef YB_HOSTSIM
  if (v > *a) *a = v;
#else
  atomicMax(a, v);
#endif
}

// min / max of a box into the box at `mn` / `mx`, one set of atomics per group of lanes of the warp that share the
// target (`key`): in the first levels a warp's 32 triangles all belong to one node, and a million lanes would queue
// on six addresses.  The float order is carried through the warp reduction as an order-preserving unsigned key.
YB_DEV uint32_t orderedKey(float v) {
  const uint32_t u = __float_as_uint(v);
  return (u >> 31) ? ~u : (u | 0x80000000u);
}
YB_DEV float fromOrderedKey(uint32_t k) { return __uint_as_float((k >> 31) ? (k & 0x7fffffffu) : ~k); }
YB_DEV void foldBoxAtomic(float* mn, float* mx, const float* lo, const float* hi, const void* key) {
#ifdef YB_HOSTSIM
  (void)key;
  for (int k = 0; k < 3; k++) atomMinF(&mn[k], lo[k]), atomMaxF(&mx[k], hi[k]);
#else
  const unsigned group = __match_any_sync(__activemask(), reinterpret_cast<unsigned long long>(key));
  const bool leader = (threadIdx.x & 31) == __ffs(group) - 1;
  for (int k = 0; k < 3; k++) {
    const uint32_t a = __reduce_min_sync(group, orderedKey(lo[k])), b = __reduce_max_sync(group, orderedKey(hi[k]));
    if (leader) atomMinF(&mn[k], fromOrderedKey(a)), atomMaxF(&mx[k], fromOrderedKey(b));
  }
#endif
}

// uint32_t(float) as x86-64 g++ evaluates it (cvttss2si to 64 bits, low word; NaN and out-of-range give 0)
YB_DEV uint32_t toU32(float x) {
  if (!(fabsf(x) < 9223372036854775808.0f)) return 0u;
  return uint32_t(uint64_t(int64_t(x)));
}
YB_DEV float halfArea(const float* mn, const float* mx) {  // bounds.hpp:38-41
  const float sx = mx[0] - mn[0], sy = mx[1] - mn[1], sz = mx[2] - mn[2];
  return sx * sy + sy * sz + sz * sx;
}
YB_DEV void emptyBox(float* mn, float* mx) {
  for (int k = 0; k < 3; k++) mn[k] = __uint_as_float(0x7f800000u), mx[k] = __uint_as_float(0xff800000u);
}
// `m < n ? m : n` folds (math_base.hpp:85-92) over finite values
YB_DEV void foldBox(float* mn, float* mx, const float* bmn, const float* bmx) {
  for (int k = 0; k < 3; k++) {
    mn[k] = mn[k] < bmn[k] ? mn[k] : bmn[k];
    mx[k] = mx[k] > bmx[k] ? mx[k] : bmx[k];
  }
}
YB_DEV uint32_t binOf(float c, float bmin, float scale) {
  const uint32_t b = toU32(scale * (c - bmin));
  return b < kBins - 1 ? b : kBins - 1;
}

// SahBVH::getSplit's cost scan (bvh.hpp:300-346) for one axis over filled bins; updates the running minimum.
YB_DEV void scanAxis(const Bin* bins, uint32_t a, float bmin, float bsize, float& minCost, uint32_t& axis, float& splitPos) {
  constexpr uint32_t nSplits = kBins - 1;
  float costs[nSplits];
  for (uint32_t i = 0; i < nSplits; i++) costs[i] = 0.0f;
  uint32_t countBelow = 0;
  float bmn[3], bmx[3];
  emptyBox(bmn, bmx);
  for (uint32_t i = 0; i < nSplits; i++) {
    float j0[3], j1[3];  // Bounds::join starts from the empty box and folds both arguments in
    emptyBox(j0, j1);
    foldBox(j0, j1, bmn, bmx);
    foldBox(j0, j1, bins[i].mn, bins[i].mx);
    for (int k = 0; k < 3; k++) bmn[k] = j0[k], bmx[k] = j1[k];
    countBelow += bins[i].count;
    costs[i] += float(countBelow) * halfArea(bmn, bmx);  // empty box: 0 * inf = NaN, never the minimum
  }
  uint32_t countAbove = 0;
  emptyBox(bmn, bmx);
  for (uint32_t i = nSplits; i > 0; i--) {
    float j0[3], j1[3];
    emptyBox(j0, j1);
    foldBox(j0, j1, bmn, bmx);
    foldBox(j0, j1, bins[i].mn, bins[i].mx);
    for (int k = 0; k < 3; k++) bmn[k] = j0[k], bmx[k] = j1[k];
    countAbove += bins[i].count;
    costs[i - 1] += float(countAbove) * halfArea(bmn, bmx);
  }
  for (uint32_t i = 0; i < nSplits; i++) {
    if (costs[i] < minCost) {
      minCost = costs[i];
      axis = a;
      splitPos = bmin + bsize * (float(i + 1) / float(kBins));
    }
  }
}
YB_DEV bool keepSplit(uint32_t span, const float* mn, const float* mx, float minCost) {
  const float leafCost = (float(span) - 0.5f) * halfArea(mn, mx);
  return !(span <= kMaxLeaf && leafCost < minCost);
}

struct Arrays {
  const float* triB;   // [n][6] padded triangle boxes
  const float* cen;    // [n][3] centroids
  uint32_t* idx;       // current order
  uint32_t* idxNext;   // order after this level's partitions
  uint32_t* nodeOf;    // position -> slot in the level's work list, kNone outside active nodes
  GNode* pool;
  uint32_t* poolCount;
  NodeWork* work;
  Bin* bins;           // [slot][3][kBins]
  unsigned long long* scan;  // inclusive counts per position: left in the high word, right in the low word
  uint32_t* tabR;      // front index of the k-th right element of the node, at [first + k - 1]
  uint32_t* tabL;      // back index of the k-th left element from the back, at [first + k - 1]
  uint32_t* nextWork;  // pool indices of the next level's active nodes
  uint32_t* nextCount;
  uint32_t* small;     // pool indices of small-subtree roots
  uint32_t* smallCount;
  uint32_t* depth;     // per pool node
  uint32_t* maxDepth;
};

// ---- stages --------------------------------------------------------------------------
struct TriPrepK {  // bvh.hpp:105-109 (fromPoints of the three vertices, padded), primitives.hpp:46 (centroid)
  const float* positions;
  const uint32_t* faces;  // stride 4
  float* triB;
  float* cen;
  YB_DEV void operator()(uint32_t i) const {
    const float* v0 = positions + 3 * size_t(faces[4 * size_t(i) + 0]);
    const float* v1 = positions + 3 * size_t(faces[4 * size_t(i) + 1]);
    const float* v2 = positions + 3 * size_t(faces[4 * size_t(i) + 2]);
    float mn[3], mx[3];
    emptyBox(mn, mx);
    const float* vs[3] = {v0, v1, v2};
    for (int p = 0; p < 3; p++)
      for (int k = 0; k < 3; k++) {
        if (vs[p][k] < mn[k]) mn[k] = vs[p][k];
        if (vs[p][k] > mx[k]) mx[k] = vs[p][k];
      }
    const float pad = float(0.001);
    for (int k = 0; k < 3; k++) {
      triB[6 * size_t(i) + k] = mn[k] - pad;
      triB[6 * size_t(i) + 3 + k] = mx[k] + pad;
      cen[3 * size_t(i) + k] = ((v0[k] + v1[k]) + v2[k]) / 3.0f;
    }
  }
};

struct RootBoundsK {  // per triangle: the root's box
  Arrays a;
  YB_DEV void operator()(uint32_t p) const {
    GNode& n = a.pool[0];
    const float* b = a.triB + 6 * size_t(a.idx[p]);
    foldBoxAtomic(n.mn, n.mx, b, b + 3, &n);
  }
};

struct WorkInitK {  // per active node
  Arrays a;
  const uint32_t* list;
  YB_DEV void operator()(uint32_t s) const {
    NodeWork& w = a.work[s];
    w.node = list[s];
    emptyBox(w.cmn, w.cmx);
    w.split = 0, w.axis = 0, w.splitPos = 0.0f, w.nLeft = 0;
    Bin* b = a.bins + size_t(s) * 3 * kBins;
    for (uint32_t i = 0; i < 3 * kBins; i++) {
      b[i].count = 0;
      emptyBox(b[i].mn, b[i].mx);
    }
  }
};
struct CentroidBoundsK {  // per position
  Arrays a;
  YB_DEV void operator()(uint32_t p) const {
    const uint32_t s = a.nodeOf[p];
    if (s == kNone) return;
    NodeWork& w = a.work[s];
    const float* c = a.cen + 3 * size_t(a.idx[p]);
    foldBoxAtomic(w.cmn, w.cmx, c, c, &w);
  }
};
struct BinK {  // per position: the three axes' bins (bvh.hpp:288-298)
  Arrays a;
  YB_DEV void operator()(uint32_t p) const {
    const uint32_t s = a.nodeOf[p];
    if (s == kNone) return;
    const NodeWork& w = a.work[s];
    const uint32_t t = a.idx[p];
    const float* c = a.cen + 3 * size_t(t);
    const float* tb = a.triB + 6 * size_t(t);
    for (uint32_t ax = 0; ax < 3; ax++) {
      const float bmin = w.cmn[ax], bsize = w.cmx[ax] - w.cmn[ax];
      const float scale = float(kBins) / bsize;
      Bin& b = a.bins[(size_t(s) * 3 + ax) * kBins + binOf(c[ax], bmin, scale)];
      atomAddU(&b.count, 1u);
      for (int k = 0; k < 3; k++) atomMinF(&b.mn[k], tb[k]), atomMaxF(&b.mx[k], tb[3 + k]);
    }
  }
};
#ifndef YB_HOSTSIM
// BinK with the bins of the block's first node in shared memory: in the first levels all 256 positions of a block
// belong to one node, and its 60 bins take the block's 256 x 21 atomics in shared memory instead of in L2.
constexpr int kBinBlock = 256;
__global__ void __launch_bounds__(kBinBlock) binSharedK(Arrays a, uint32_t n) {
  __shared__ uint32_t sCount[3 * kBins];
  __shared__ float sMn[3 * kBins][3], sMx[3 * kBins][3];
  const uint32_t p = blockIdx.x * kBinBlock + threadIdx.x;
  const uint32_t blockSlot = a.nodeOf[blockIdx.x * kBinBlock];
  if (threadIdx.x < 3 * kBins) {
    sCount[threadIdx.x] = 0;
    emptyBox(sMn[threadIdx.x], sMx[threadIdx.x]);
  }
  __syncthreads();
  const uint32_t s = p < n ? a.nodeOf[p] : kNone;
  if (s != kNone) {
    const NodeWork& w = a.work[s];
    const uint32_t t = a.idx[p];
    const float* c = a.cen + 3 * size_t(t);
    const float* tb = a.triB + 6 * size_t(t);
    for (uint32_t ax = 0; ax < 3; ax++) {
      const float bmin = w.cmn[ax], bsize = w.cmx[ax] - w.cmn[ax];
      const float scale = float(kBins) / bsize;
      const uint32_t bi = ax * kBins + binOf(c[ax], bmin, scale);
      if (s == blockSlot) {
        atomicAdd(&sCount[bi], 1u);
        for (int k = 0; k < 3; k++) atomMinF(&sMn[bi][k], tb[k]), atomMaxF(&sMx[bi][k], tb[3 + k]);
      } else {
        Bin& b = a.bins[size_t(s) * 3 * kBins + bi];
        atomicAdd(&b.count, 1u);
        for (int k = 0; k < 3; k++) atomMinF(&b.mn[k], tb[k]), atomMaxF(&b.mx[k], tb[3 + k]);
      }
    }
  }
  __syncthreads();
  if (threadIdx.x < 3 * kBins && blockSlot != kNone && sCount[threadIdx.x] > 0) {
    Bin& b = a.bins[size_t(blockSlot) * 3 * kBins + threadIdx.x];
    atomicAdd(&b.count, sCount[threadIdx.x]);
    for (int k = 0; k < 3; k++) atomMinF(&b.mn[k], sMn[threadIdx.x][k]), atomMaxF(&b.mx[k], sMx[threadIdx.x][k]);
  }
}
#endif

struct ChooseK {  // per active node: SahBVH::getSplit's decision
  Arrays a;
  YB_DEV void operator()(uint32_t s) const {
    NodeWork& w = a.work[s];
    const GNode& n = a.pool[w.node];
    float minCost = __uint_as_float(0x7f800000u);
    uint32_t axis = 0;
    float splitPos = 0.0f;
    for (uint32_t ax = 0; ax < 3; ax++)
      scanAxis(a.bins + (size_t(s) * 3 + ax) * kBins, ax, w.cmn[ax], w.cmx[ax] - w.cmn[ax], minCost, axis, splitPos);
    w.split = keepSplit(n.span, n.mn, n.mx, minCost) ? 1u : 0u;
    w.axis = axis, w.splitPos = splitPos;
  }
};
struct ClassK {  // per position: class of the element under its node's split (left in the high word)
  Arrays a;
  YB_DEV void operator()(uint32_t p) const {
    unsigned long long v = 0ull;
    const uint32_t s = a.nodeOf[p];
    if (s != kNone && a.work[s].split) {
      const NodeWork& w = a.work[s];
      const bool left = a.cen[3 * size_t(a.idx[p]) + w.axis] < w.splitPos;
      v = left ? (1ull << 32) : 1ull;
    }
    a.scan[p] = v;
  }
};
// counts relative to the node: inclusive prefix at p minus the inclusive prefix just before the node
YB_DEV void nodeCounts(const Arrays& a, uint32_t first, uint32_t p, uint32_t& inclL, uint32_t& inclR) {
  const unsigned long long base = first ? a.scan[first - 1] : 0ull, v = a.scan[p] - base;
  inclL = uint32_t(v >> 32), inclR = uint32_t(v);
}
struct TablesK {  // per position of a splitting node
  Arrays a;
  YB_DEV void operator()(uint32_t p) const {
    const uint32_t s = a.nodeOf[p];
    if (s == kNone || !a.work[s].split) return;
    const GNode& n = a.pool[a.work[s].node];
    uint32_t inclL, inclR, totL, totR;
    nodeCounts(a, n.first, p, inclL, inclR);
    nodeCounts(a, n.first, n.first + n.span - 1, totL, totR);
    const bool left = a.cen[3 * size_t(a.idx[p]) + a.work[s].axis] < a.work[s].splitPos;
    const uint32_t f = p - n.first;
    if (!left) a.tabR[n.first + inclR - 1] = f;                              // the inclR-th right element from the front
    else a.tabL[n.first + (totL - inclL + 1) - 1] = n.span - 1 - f;          // the (totL - inclL + 1)-th left from the back
    if (f == 0) a.work[s].nLeft = totL;
  }
};
struct PartitionK {  // per position: where the reference's in-place partition leaves this element
  Arrays a;
  YB_DEV void operator()(uint32_t p) const {
    const uint32_t s = a.nodeOf[p];
    if (s == kNone || !a.work[s].split) {
      a.idxNext[p] = a.idx[p];
      return;
    }
    const GNode& n = a.pool[a.work[s].node];
    const uint32_t first = n.first, span = n.span, last = first + span - 1;
    uint32_t inclL, inclR, totL, totR;
    nodeCounts(a, first, p, inclL, inclR);
    nodeCounts(a, first, last, totL, totR);
    const bool left = a.cen[3 * size_t(a.idx[p]) + a.work[s].axis] < a.work[s].splitPos;
    const uint32_t f = p - first, b = span - 1 - f;
    const uint32_t kR = inclR - (left ? 0u : 1u);  // right elements before f in the front stream
    const uint32_t lF = f - kR;                    // left elements before f
    // back elements examined before front element f: through the kR-th left element of the back stream
    unsigned long long bc = 0ull;
    if (kR > 0) bc = kR <= totL ? (unsigned long long)a.tabL[first + kR - 1] + 1ull : (unsigned long long)span + 1ull;
    uint32_t dest;
    if ((unsigned long long)f + bc <= (unsigned long long)(span - 1)) {
      dest = left ? first + lF + kR : last - uint32_t(bc);
    } else {
      // examined from the back: in back run r, which starts when the r-th right element of the front stream was found
      const uint32_t lB = totL - inclL;  // left elements behind p = before b in the back stream
      const uint32_t r = lB + 1;
      dest = left ? first + a.tabR[first + r - 1] : last - (b + 1);
    }
    a.idxNext[dest] = a.idx[p];
  }
};
struct ChildrenK {  // per active node: bvh.hpp:160-183
  Arrays a;
  YB_DEV void operator()(uint32_t s) const {
    const NodeWork& w = a.work[s];
    GNode& n = a.pool[w.node];
    if (!w.split || w.nLeft == 0 || w.nLeft == n.span) return;  // stays a leaf (its indices keep the partition's order)
    const uint32_t l = atomAddU(a.poolCount, 2u);
    n.left = l;
    atomMaxU(a.maxDepth, a.depth[w.node] + 1u);
    for (uint32_t c = 0; c < 2; c++) {
      GNode& ch = a.pool[l + c];
      emptyBox(ch.mn, ch.mx);
      ch.first = c == 0 ? n.first : n.first + w.nLeft;
      ch.span = c == 0 ? w.nLeft : n.span - w.nLeft;
      ch.left = 0, ch.slot = kNone;
      a.depth[l + c] = a.depth[w.node] + 1u;
      if (ch.span > kSmallSpan) {
        ch.slot = atomAddU(a.nextCount, 1u);
        a.nextWork[ch.slot] = l + c;
      } else {
        a.small[atomAddU(a.smallCount, 1u)] = l + c;
      }
    }
  }
};
struct ChildBoundsK {  // per position (new order): updateBounds of the two children; the position's slot in the next level
  Arrays a;
  YB_DEV void operator()(uint32_t p) const {
    const uint32_t s = a.nodeOf[p];
    if (s == kNone) return;
    const NodeWork& w = a.work[s];
    const GNode& n = a.pool[w.node];
    if (n.left == 0) {
      a.nodeOf[p] = kNone;
      return;
    }
    GNode& ch = a.pool[n.left + (p < n.first + w.nLeft ? 0u : 1u)];
    a.nodeOf[p] = ch.slot;
    const float* tb = a.triB + 6 * size_t(a.idxNext[p]);
    foldBoxAtomic(ch.mn, ch.mx, tb, tb + 3, &ch);
  }
};
// One thread finishes a small subtree with the reference's sequential code (bvh.hpp:140-184, 273-347).
struct SmallSubtreeK {
  Arrays a;
  YB_DEV void operator()(uint32_t s) const {
    uint32_t stack[64];
    int sp = 0;
    stack[sp++] = a.small[s];
    while (sp > 0) {
      const uint32_t self = stack[--sp];
      GNode& n = a.pool[self];
      const uint32_t first = n.first, span = n.span;
      // getSplit
      float cmn[3], cmx[3];
      emptyBox(cmn, cmx);
      for (uint32_t i = first; i < first + span; i++) {
        const float* c = a.cen + 3 * size_t(a.idx[i]);
        for (int k = 0; k < 3; k++) {
          cmn[k] = cmn[k] < c[k] ? cmn[k] : c[k];
          cmx[k] = cmx[k] > c[k] ? cmx[k] : c[k];
        }
      }
      float minCost = __uint_as_float(0x7f800000u), splitPos = 0.0f;
      uint32_t axis = 0;
      for (uint32_t ax = 0; ax < 3; ax++) {
        Bin bins[kBins];
        for (uint32_t i = 0; i < kBins; i++) {
          bins[i].count = 0;
          emptyBox(bins[i].mn, bins[i].mx);
        }
        const float bmin = cmn[ax], bsize = cmx[ax] - cmn[ax];
        const float scale = float(kBins) / bsize;
        for (uint32_t i = first; i < first + span; i++) {
          const uint32_t t = a.idx[i];
          Bin& b = bins[binOf(a.cen[3 * size_t(t) + ax], bmin, scale)];
          b.count++;
          foldBox(b.mn, b.mx, a.triB + 6 * size_t(t), a.triB + 6 * size_t(t) + 3);
        }
        scanAxis(bins, ax, bmin, bsize, minCost, axis, splitPos);
      }
      if (!keepSplit(span, n.mn, n.mx, minCost)) continue;
      // the in-place partition
      long long i = first, j = (long long)first + span - 1;
      while (i <= j) {
        if (a.cen[3 * size_t(a.idx[i]) + axis] < splitPos) {
          i++;
        } else {
          const uint32_t t = a.idx[i];
          a.idx[i] = a.idx[j];
          a.idx[j] = t;
          j--;
        }
      }
      const uint32_t nLeft = uint32_t(i - first);
      if (nLeft == 0 || nLeft == span) continue;
      const uint32_t l = atomAddU(a.poolCount, 2u);
      n.left = l;
      atomMaxU(a.maxDepth, a.depth[self] + 1u);
      for (uint32_t c = 0; c < 2; c++) {
        GNode& ch = a.pool[l + c];
        a.depth[l + c] = a.depth[self] + 1u;
        ch.first = c == 0 ? first : first + nLeft;
        ch.span = c == 0 ? nLeft : span - nLeft;
        ch.left = 0, ch.slot = kNone;
        emptyBox(ch.mn, ch.mx);
        for (uint32_t q = ch.first; q < ch.first + ch.span; q++)
          foldBox(ch.mn, ch.mx, a.triB + 6 * size_t(a.idx[q]), a.triB + 6 * size_t(a.idx[q]) + 3);
      }
      // the reference recurses into the left child first; the order does not matter here (disjoint ranges)
      if (sp + 2 <= 64) stack[sp++] = l + 1, stack[sp++] = l;
    }
  }
};


// ---- the reference's node numbering ----------------------------------------------------------------------------------
// BVH::subdivide numbers a node's two children when the node is visited, depth first, left subtree first (bvh.hpp:165-166,
// 180-183): the children of the inner node with pre-order rank p (among inner nodes) are 1 + 2 p and 2 + 2 p.  The pool is
// in creation order with child links; inner-node counts per subtree come bottom-up, ranks top-down, one depth at a time.
struct RefNode {  // = RefBvhNode of the host layer, the reference's BVHNode (bvh.hpp:21-33)
  float mn[3], mx[3];
  uint32_t leftFirst, span;
};
struct CountUpK {
  Arrays a;
  uint32_t* cnt;
  uint32_t d;
  YB_DEV void operator()(uint32_t i) const {
    if (a.depth[i] != d) return;
    const uint32_t l = a.pool[i].left;
    cnt[i] = l ? 1u + cnt[l] + cnt[l + 1] : 0u;
  }
};
struct NumberDownK {
  Arrays a;
  const uint32_t* cnt;
  uint32_t *pre, *ref;
  uint32_t d;
  YB_DEV void operator()(uint32_t i) const {
    if (a.depth[i] != d) return;
    const uint32_t l = a.pool[i].left;
    if (!l) return;
    const uint32_t p = pre[i], r = 1u + 2u * p;
    ref[l] = r, ref[l + 1] = r + 1u;
    pre[l] = p + 1u, pre[l + 1] = p + 1u + cnt[l];
  }
};
struct EmitK {
  Arrays a;
  const uint32_t *pre, *ref;
  RefNode* out;
  YB_DEV void operator()(uint32_t i) const {
    const GNode& g = a.pool[i];
    RefNode o;
    for (int k = 0; k < 3; k++) o.mn[k] = g.mn[k], o.mx[k] = g.mx[k];
    if (g.left) o.leftFirst = 1u + 2u * pre[i], o.span = 0u;
    else o.leftFirst = g.first, o.span = g.span;
    out[ref[i]] = o;
  }
};


// One device allocation, handed out in 256-byte-aligned pieces (pass 1: sizes only, base == nullptr).
struct Arena {
  char* base = nullptr;
  size_t used = 0;
  ~Arena() { rt::release(base); }
  template <class T>
  T* take(size_t count) {
    used = (used + 255) & ~size_t(255);
    T* p = base ? reinterpret_cast<T*>(base + used) : nullptr;
    used += count * sizeof(T);
    return p;
  }
};

// ---- the build ------------------------------------------------------------------------------
// Returns nullptr or an error string.  `nodesOut` receives up to 2 n nodes in the reference's numbering, `indicesOut` the
// reference's m_indices.
inline const char* build(rt::Stream& st, const float* positions, size_t nVerts, const uint32_t* faces4, size_t nTris,
                         RefNode* nodesOut, uint32_t* nNodesOut, uint32_t* indicesOut, uint32_t* levelsOut) {
  if (nTris == 0 || nTris > 0x7ffffff0u) return "triangle count out of range";
  const uint32_t n = uint32_t(nTris);
  // one device allocation for everything (18 cudaMalloc / cudaFree pairs cost more than the build itself)
  const size_t maxActive = size_t(n) / (kSmallSpan + 1) + 2;  // active nodes are disjoint runs of more than kSmallSpan
  Arena arena;
#define YB_B(expr)                       \
  do {                                   \
    if (const char* e_ = (expr)) return e_; \
  } while (0)
  float *dPos = nullptr, *triB = nullptr, *cen = nullptr;
  uint32_t *dFaces = nullptr, *idxA = nullptr, *idxB = nullptr, *nodeOf = nullptr, *counters = nullptr, *listA = nullptr, *listB = nullptr,
           *small = nullptr, *tabR = nullptr, *tabL = nullptr;
  GNode* pool = nullptr;
  NodeWork* work = nullptr;
  Bin* bins = nullptr;
  unsigned long long *scan = nullptr, *sums = nullptr;
  uint32_t *depth = nullptr, *cnt = nullptr, *pre = nullptr, *ref = nullptr;
  RefNode* refNodes = nullptr;
  for (int pass = 0; pass < 2; pass++) {  // pass 0 sizes the arena, pass 1 hands out the pieces
    arena.used = 0;
    dPos = arena.take<float>(3 * nVerts), dFaces = arena.take<uint32_t>(4 * size_t(n));
    triB = arena.take<float>(6 * size_t(n)), cen = arena.take<float>(3 * size_t(n));
    idxA = arena.take<uint32_t>(n), idxB = arena.take<uint32_t>(n), nodeOf = arena.take<uint32_t>(n);
    tabR = arena.take<uint32_t>(n), tabL = arena.take<uint32_t>(n);
    scan = arena.take<unsigned long long>(n), sums = arena.take<unsigned long long>(size_t(n) / 1024 + 64);
    pool = arena.take<GNode>(2 * size_t(n) + 2);
    work = arena.take<NodeWork>(maxActive), bins = arena.take<Bin>(maxActive * 3 * kBins);
    listA = arena.take<uint32_t>(maxActive), listB = arena.take<uint32_t>(maxActive);
    small = arena.take<uint32_t>(size_t(n) + 2), counters = arena.take<uint32_t>(4);
    depth = arena.take<uint32_t>(2 * size_t(n) + 2), cnt = arena.take<uint32_t>(2 * size_t(n) + 2);
    pre = arena.take<uint32_t>(2 * size_t(n) + 2), ref = arena.take<uint32_t>(2 * size_t(n) + 2);
    refNodes = arena.take<RefNode>(2 * size_t(n) + 2);
    if (pass == 0) {
      void* v = nullptr;
      YB_B(rt::alloc(&v, arena.used + 256));
      arena.base = static_cast<char*>(v);
    }
  }
  // YART_B200_BUILD_TRACE=1: stage times on stderr
  const char* traceEnv = getenv("YART_B200_BUILD_TRACE");
  const bool trace = traceEnv && *traceEnv && *traceEnv != '0';
  auto now = [] { return std::chrono::high_resolution_clock::now(); };
  auto msSince = [&](std::chrono::high_resolution_clock::time_point t) {
    rt::sync(st);
    return std::chrono::duration<double, std::milli>(now() - t).count();
  };
  const auto t0 = now();
  double tAlloc = 0, tPrep = 0, tLevels = 0, tSmall = 0;
  if (trace) tAlloc = msSince(t0);
  YB_B(rt::h2d(st, dPos, positions, 3 * nVerts * sizeof(float)));
  YB_B(rt::h2d(st, dFaces, faces4, 4 * size_t(n) * sizeof(uint32_t)));

  // init (bvh.hpp:41-67): identity order, the root over everything
  std::vector<uint32_t> iota(n);
  for (uint32_t i = 0; i < n; i++) iota[i] = i;
  YB_B(rt::h2d(st, idxA, iota.data(), size_t(n) * sizeof(uint32_t)));
  GNode root{};
  for (int k = 0; k < 3; k++) root.mn[k] = std::numeric_limits<float>::infinity(), root.mx[k] = -std::numeric_limits<float>::infinity();
  root.first = 0, root.span = n, root.left = 0, root.slot = kNone;
  YB_B(rt::h2d(st, pool, &root, sizeof root));
  uint32_t hc[4] = {1u, 0u, 0u, 0u};
  YB_B(rt::h2d(st, counters, hc, sizeof hc));
  rt::launchFor(st, n, TriPrepK{dPos, dFaces, triB, cen});

  Arrays a{};
  a.triB = triB, a.cen = cen, a.idx = idxA, a.idxNext = idxB, a.nodeOf = nodeOf, a.pool = pool, a.poolCount = counters;
  a.work = work, a.bins = bins, a.scan = scan, a.tabR = tabR, a.tabL = tabL, a.nextWork = listB, a.nextCount = counters + 1;
  a.small = small, a.smallCount = counters + 2;
  a.depth = depth, a.maxDepth = counters + 3;
  YB_B(rt::zero(st, depth, sizeof(uint32_t)));  // the root
  rt::launchFor(st, n, RootBoundsK{a});
  if (trace) tPrep = msSince(t0);
  uint32_t* list = listA;
  uint32_t nActive = 0, levels = 0;
  if (n > kSmallSpan) {
    const uint32_t zero = 0;
    YB_B(rt::h2d(st, listA, &zero, sizeof zero));
    YB_B(rt::zero(st, nodeOf, size_t(n) * sizeof(uint32_t)));  // every position in slot 0
    nActive = 1;
  } else {
    const uint32_t zero = 0, one = 1;
    YB_B(rt::h2d(st, small, &zero, sizeof zero));
    YB_B(rt::h2d(st, counters + 2, &one, sizeof one));
  }
  while (nActive > 0) {
    if (++levels > 4096) return "BVH build does not terminate";
    if (nActive > maxActive) return "BVH build: too many active nodes";
    a.nextWork = list == listA ? listB : listA;
    rt::launchFor(st, nActive, WorkInitK{a, list});
    rt::launchFor(st, n, CentroidBoundsK{a});
#ifdef YB_HOSTSIM
    rt::launchFor(st, n, BinK{a});
#else
    binSharedK<<<(n + kBinBlock - 1) / kBinBlock, kBinBlock, 0, st.s>>>(a, n);
#endif
    rt::launchFor(st, nActive, ChooseK{a});
    rt::launchFor(st, n, ClassK{a});
    inclusiveScan(st, scan, sums, n);
    rt::launchFor(st, n, TablesK{a});
    rt::launchFor(st, n, PartitionK{a});
    rt::launchFor(st, nActive, ChildrenK{a});
    rt::launchFor(st, n, ChildBoundsK{a});
    YB_B(rt::d2h(st, hc, counters, sizeof hc));
    nActive = hc[1];
    hc[1] = 0;
    YB_B(rt::h2d(st, counters + 1, &hc[1], sizeof(uint32_t)));
    list = a.nextWork;
    uint32_t* t = a.idx;
    a.idx = a.idxNext, a.idxNext = t;
  }
  YB_B(rt::d2h(st, hc, counters, sizeof hc));
  if (trace) tLevels = msSince(t0);
  const uint32_t nSmall = hc[2];
  if (hc[2] > 0) rt::launchFor(st, hc[2], SmallSubtreeK{a});
  YB_B(rt::d2h(st, hc, counters, sizeof hc));
  if (const char* e = rt::lastError()) return e;
  if (trace) tSmall = msSince(t0);
  if (hc[0] > 2 * n + 2) return "BVH build: node pool overflow";
  {
    const uint32_t nNodes = hc[0], deepest = hc[3];
    if (deepest > 4096) return "BVH build: tree too deep";
    for (uint32_t d = deepest + 1; d-- > 0;) rt::launchFor(st, nNodes, CountUpK{a, cnt, d});
    YB_B(rt::zero(st, pre, sizeof(uint32_t)));
    YB_B(rt::zero(st, ref, sizeof(uint32_t)));
    for (uint32_t d = 0; d <= deepest; d++) rt::launchFor(st, nNodes, NumberDownK{a, cnt, pre, ref, d});
    rt::launchFor(st, nNodes, EmitK{a, pre, ref, refNodes});
  }
  YB_B(rt::d2h(st, nodesOut, refNodes, size_t(hc[0]) * sizeof(RefNode)));
  YB_B(rt::d2h(st, indicesOut, a.idx, size_t(n) * sizeof(uint32_t)));
  *nNodesOut = hc[0];
  if (levelsOut) *levelsOut = levels;
  if (trace)
    fprintf(stderr, "yart_b200 bvh build: %u tris, alloc %.1f ms, upload + prep %.1f, %u levels %.1f, %u small subtrees %.1f, download %.1f; %u nodes\n",
            n, tAlloc, tPrep - tAlloc, levels, tLevels - tPrep, nSmall, tSmall - tLevels, msSince(t0) - tSmall, hc[0]);
#undef YB_B
  return nullptr;
}

}  // namespace bvhb
}  // namespace yb
