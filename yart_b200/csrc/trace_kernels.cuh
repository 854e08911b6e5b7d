// trace_kernels.cuh — persistent-warp traversal engine (CUDA only) shared by the extend, shadow and
// ray-hook kernels of both BVH layouts: the reference-order BVH2 (Bvh2Walk, traverse.cuh) and the 4-wide
// quantised BVH (WideWalk, wide_bvh.cuh).  The layout type supplies the box test, the mesh's nodes, the
// inner-node step and whether leaves are parked; everything else below is shared.
//
// With Bvh2Walk every ray performs exactly the reference's sequence of box and triangle tests
// (RayIntegrator::testNode / testBVH / testTriangle, src/cpu/ray-integrator.cpp:20-229, through the
// arithmetic in traverse.cuh); what changes is only how the 32 lanes of a warp are kept busy:
//   * each lane is a small state machine: IDLE → NODE (scene-graph node set-up) → TRAV (inside one
//     mesh's BVH: current ref is an inner node or a leaf) → … → IDLE;
//   * idle lanes are refilled from the work queue with ONE atomic per warp (ballot + popc), as soon
//     as enough lanes are idle, instead of waiting for the slowest ray of a batch of 32;
//   * inner-node steps run in a tight loop while enough lanes sit on inner nodes; a lane that reaches a
//     leaf parks it and keeps walking (its own test order is unchanged: parked leaves are tested in the
//     order they were reached, before any later leaf), and all leaves are processed together, so the two
//     code paths do not serialise against each other on every iteration;
//   * the inner step is branch-free apart from its `inner` guard: packed (ref, d) stack entries in shared
//     memory ([entry][thread], conflict-free, one LDS.64 / STS.64 per pop / push), the stack pointer is
//     the shared byte address, a sentinel at the bottom replaces the "empty" test, one predicated pop
//     site per iteration, descend / push as selects; trees deeper than kShStack spill to global memory
//     through an out-of-line path; no local memory is used.
// Node records are fetched as two 256-bit read-only loads, triangles as three 128-bit loads.
// With WideWalk the set of boxes differs, the triangle arithmetic does not (wide_bvh.cuh's header).
#pragma once
#include "integrator.cuh"

namespace yb {

// Ray in the object space of scene node `node`: the chain of inverse transforms root → node, applied
// in the recursion's order (ray-integrator.cpp:26-30).  The ancestor chain is a host-built table.
__device__ __forceinline__ void nodeLocalRay(const DScene& sc, uint32_t node, int depth, V3& o, V3& d) {
  const int32_t* __restrict__ path = sc.nodePath + size_t(node) * YC_MAX_NODE_DEPTH;
#pragma unroll 1
  for (int level = 0; level <= depth; level++) {
    const YcNode& nd = sc.nodes[path[level]];
    const V3 no = xformRows(nd.inv, o, 1.0f), ndir = xformRows(nd.inv, d, 0.0f);
    o = no;
    d = ndir;
  }
}

enum : int { kLaneIdle = 0, kLaneNode = 1, kLaneTrav = 2 };

// IO policy:  bool load(uint32_t j, V3& o, V3& d, float& tMax, Sampler& smp)   (false: nothing to trace)
//             void store(uint32_t j, const TraceState& st, bool didHit, const Sampler& smp)
// EARLY_OUT (NEE only): a lane stops at its first accepted occluder.
template <class Walk, bool NEE, bool ALPHA, bool COUNT, bool EARLY_OUT, class IO>
__device__ __forceinline__ void tracePersistent(const DScene& sc, IO& io, uint32_t n, uint32_t* head, uint2* spillBase,
                                                const TraceTuning tune, TraceCounters& cnt) {
  __shared__ uint2 shStack[kPsStack * kTraceBlock];
  __shared__ uint2* shSpill;
  WarpStack stack;
  stack.init(shStack, &shSpill, spillBase, tune.shEntries);
  const unsigned FULL = 0xffffffffu;
  const unsigned lane = threadIdx.x & 31u, ltMask = (1u << lane) - 1u;

  int state = kLaneIdle;
  bool exhausted = false;
  uint32_t item = 0, nextNode = 0, cur = 0;
  uint32_t sp = 0;  // stack pointer: shared byte address of the next free slot (WarpStack)
  int curNode = 0;
  float dcur = 0.0f;
  bool didHit = false, meshHit = false, rayIsWorld = false, worldFinite = false;
  V3 wo, wd;
  typename Walk::Ray r;
  TraceState st;
  Sampler smp;
  const float4* __restrict__ nodes = nullptr;
  const float4* __restrict__ tris = nullptr;
  uint32_t meshIdx = 0;
  constexpr bool SPEC = Walk::parks(COUNT);
  uint32_t pend = 0u;                     // parked leaf (0 = none; leaf refs carry bit 31)
  float pendD = 0.0f;

  for (;;) {
    // ---- refill idle lanes -------------------------------------------------------------------
    const unsigned idle = __ballot_sync(FULL, state == kLaneIdle);
    if (idle) {
      if (!exhausted && (__popc(idle) >= tune.refillMin || idle == FULL)) {
        const uint32_t want = uint32_t(__popc(idle));
        uint32_t base = 0;
        if (lane == 0) base = atomicAdd(head, want);
        base = __shfl_sync(FULL, base, 0);
        if (state == kLaneIdle) {
          const uint32_t j = base + uint32_t(__popc(idle & ltMask));
          if (j < n) {
            float tMax;
            if (io.load(j, wo, wd, tMax, smp)) {
              item = j;
              rayIsWorld = false;
              worldFinite = isfinite(wo.x) && isfinite(wo.y) && isfinite(wo.z) && isfinite(wd.x) && isfinite(wd.y) &&
                            isfinite(wd.z);
              initTraceState(st, tMax);
              nextNode = 0;
              didHit = false;
              state = kLaneNode;
            }
          }
        }
        if (base + want >= n) exhausted = true;
      }
      if (exhausted && __ballot_sync(FULL, state != kLaneIdle) == 0) break;
    }

    // ---- scene-graph step: find the next node whose box the ray enters (testNode) ------------------
    if (state == kLaneNode) {
      bool entered = false;
      while (nextNode < sc.nNodes) {
        const YcNode& nd = sc.nodes[nextNode];
        if (nd.identityChain && worldFinite) {
          // every transform from the root to this node is exactly the identity: the matrix products
          // ((0 + 1*x) + 0*y + 0*z) + 0*w reduce to x + 0 for finite inputs (-0 becomes +0), so the
          // local ray is the canonicalised world ray — computed once per ray and kept.
          if (!rayIsWorld) {
            r.set(wo + 0.0f, wd + 0.0f);
            rayIsWorld = true;
          }
        } else {
          V3 o = wo, d = wd;
          nodeLocalRay(sc, nextNode, nd.depth, o, d);
          r.set(o, d);
          rayIsWorld = false;
        }
        float dd;
        if (!Walk::template box<COUNT>(r, V3(nd.bmin), V3(nd.bmax), st.hit.t, dd, cnt) || st.hit.t < dd) {
          nextNode = uint32_t(nd.skip);
          continue;
        }
        const int mi = nd.mesh;
        curNode = int(nextNode);
        nextNode++;
        if (mi < 0) continue;
        const YcMesh& mesh = sc.meshes[mi];
        if (!Walk::template box<COUNT>(r, V3(mesh.rootMin), V3(mesh.rootMax), st.hit.t, dd, cnt)) continue;  // testBVH's root test
        meshIdx = uint32_t(mi);
        nodes = Walk::nodes(sc, mi, mesh);
        tris = sc.bvhTris + 3 * size_t(mesh.triOffset);
        cur = Walk::rootRef(sc, mi, mesh);
        dcur = dd;
        stack.put(stack.base, kNoRef, 0.0f);  // sentinel
        sp = stack.base + kPsStride;
        pend = 0u;
        meshHit = false;
        entered = true;
        break;
      }
      if (entered) {
        state = kLaneTrav;
      } else {
        io.store(item, st, didHit, smp);
        state = kLaneIdle;
      }
    }

    // ---- inner-node steps ------------------------------------------------------------------------
    // SPEC (Walk::parks: the wide walk always, the BVH2 walk in non-counting builds): a lane that reaches a leaf
    // parks it in `pend` and keeps walking;
    // it only blocks when it reaches a second leaf (or has walked the mesh) with one still parked.
    // Parked leaves are tested in the order they were reached, before any later leaf, so the sequence
    // of triangle tests — and with it the accepted hit, exact ties and alpha-test draws — is the
    // reference's.  Only box culling sees a slightly older hit.t, i.e. a few extra box tests.
    // The loop body is branch-free apart from the `inner` guard: descend / push / pop are selects and
    // predicated 64-bit shared-memory accesses, and the stack sentinel stands in for the "empty" test.
    for (;;) {
      const bool trav = state == kLaneTrav;
      bool doPop = trav && cur == kPopRef;  // left by the previous step: one pop site per iteration
      if (SPEC && trav && pend == 0u && int32_t(cur) < Walk::kParkBelow) {
        pend = cur, pendD = dcur;
        doPop = true;
      }
      stack.popIf(doPop, sp, cur, dcur);  // the sentinel ends the mesh: cur = kNoRef
      const bool inner = trav && int32_t(cur) >= 0;
      const unsigned im = __ballot_sync(FULL, inner);
      if (im == 0) break;
      if (__popc(im) < tune.innerMin && __ballot_sync(FULL, trav && !inner)) break;
      if (inner) Walk::template inner<COUNT>(r, nodes, st.hit.t, stack, sp, cur, dcur, tune, cnt);
    }

    // ---- leaf step -------------------------------------------------------------------------------
    // kNoRef carries the leaf bit, so "cur is a leaf" also covers "mesh walked" (with or without a
    // parked leaf); a lane still on an inner node uses the break to test its parked leaf.
    if (state == kLaneTrav && (int32_t(cur) < 0 || (SPEC && pend != 0u))) {
      uint32_t leaf = cur;
      float leafD = dcur;
      if (SPEC) {
        // a real leaf in `cur` with nothing parked cannot leave the loop above (it is parked at once)
        leaf = pend, leafD = pendD;
        pend = 0u;
      }
      // the didHit test never fails (an early-out lane goes idle at its first occluder, below); it is kept because
      // without it ptxas spills 4 more bytes in the counting wide ray-hook kernel
      if (int32_t(leaf) < -1 && leafD < st.hit.t && !(NEE && EARLY_OUT && didHit)) {
        const YcMesh& mesh = sc.meshes[meshIdx];
        uint32_t ti = leaf & ~YC_REF_LEAF;
        while (true) {
          const float4 a = __ldg(tris + 3 * size_t(ti)), b = __ldg(tris + 3 * size_t(ti) + 1),
                       c = __ldg(tris + 3 * size_t(ti) + 2);
          meshHit |= testTriangle<NEE, ALPHA, COUNT>(sc, mesh, r, a, b, c, curNode, st, &smp, cnt);
          if (NEE && meshHit) break;  // ray-integrator.cpp:121: leaves the leaf loop only
          if (__float_as_uint(c.z) & YC_TRI_LAST) break;
          ti++;
        }
        didHit |= meshHit;
      }
      if (NEE && EARLY_OUT && didHit) {
        io.store(item, st, true, smp);
        state = kLaneIdle;
        pend = 0u;
      } else {
        if (!SPEC && cur != kNoRef) stack.pop(sp, cur, dcur);
        if (cur == kNoRef) state = kLaneNode;  // mesh walked and nothing parked any more
      }
    }
  }
}

}  // namespace yb
