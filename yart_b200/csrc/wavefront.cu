// wavefront.cu — the device layer of libyart_b200.so: yc_* entry points (include/yart_cuda.h) and
// the wavefront kernels that replace yart's src/cpu tile renderer on sm_100a.
//
//   raygen → [ extend → shade → shadow ]* → accumulate   per chunk of pixel-samples
//   finalize (estimator value, wave blend, tonemap)      per wave
//
// Reference mapping: TileRenderer worker loop + finishTile (src/cpu/tile-renderer.hpp:161-191,
// 205-239), Integrator::render (src/cpu/integrator.cpp:5-28), MISIntegrator::Li/Ld
// (src/cpu/mis-integrator.cpp:13-148), RayIntegrator::testNode (src/cpu/ray-integrator.cpp:20-54).
// The per-path arithmetic lives in integrator.cuh / traverse.cuh / bsdf.cuh / lights.cuh; this file
// owns memory, queues, launch geometry and the C ABI.  Compile with -fmad=false (dmath.cuh).
//
// extend and shadow are persistent kernels: one CTA set sized to the SM count, each warp pulling
// 32 queue entries at a time with one atomic (lane 0) and keeping its traversal stack in shared
// memory; node and triangle records are read as 128-bit loads (traverse.cuh).  shade compacts the
// surviving paths and the NEE requests into the next queues with warp-aggregated appends.
#include <algorithm>
#include <cstdarg>
#include <vector>

#include "estimator.cuh"
#include "integrator.cuh"
#include "rt.cuh"
#include "comm.cuh"
#include "bvh_build.cuh"
#ifndef YB_HOSTSIM
#include "trace_kernels.cuh"
#endif

using namespace yb;

#ifndef YB_TRACE_MIN_BLOCKS
#define YB_TRACE_MIN_BLOCKS 7  // CTAs x 4 warps per SM of the reference-order closest-hit kernels: 72 registers, no spills in the alpha build (8 CTAs = 64 registers: Sponza-shaped step 28.4-28.9 ms, 7: 27.2, 6: 27.8 on one box)
#endif
#ifndef YB_SHADOW_MIN_BLOCKS
#define YB_SHADOW_MIN_BLOCKS 7  // 72 registers, no spills (uncapped: 96 registers, 5 CTAs — C2 step 11.5 ms; 7: 10.9; 8 spills: 11.9)
#endif
// Resident CTAs (x 256 threads) per SM the three shading kernels are compiled for (registers = 65536 / 256 / CTAs)
#ifndef YB_RESOLVE_MIN_BLOCKS
#define YB_RESOLVE_MIN_BLOCKS 4
#endif
#ifndef YB_SAMPLE_MIN_BLOCKS
#define YB_SAMPLE_MIN_BLOCKS 4
#endif
#ifndef YB_NEE_MIN_BLOCKS
#define YB_NEE_MIN_BLOCKS 4
#endif

// ---------------------------------------------------------------------------------------
// context
// ---------------------------------------------------------------------------------------
enum { kCtrExtendHead = 0, kCtrNextCount = 1, kCtrShadowCount = 2, kCtrShadowHead = 3, kCtrHitCount = 4,
       kCtrNeeCount = 6, kCtrCount = 8 };

// Two chunks of a wave are in flight at a time, each on its own stream with its own path state: while one
// chunk waits for the slowest ray of a traversal launch (a single ray with a zero direction component can walk
// 14 K boxes alone, see profiles/README.md) or for its bounce-count read-back, the other keeps the GPU busy.
constexpr int kLanes = 2;
struct Lane {
  rt::Stream st;       // the lane's own stream (the context's main stream runs finalize, copies, ray hooks, collectives)
  PathState ps{};      // ps.L points at Lbuf[lSel] while a chunk is in flight
  ShadowQueue sq{};
  SurfState ss{};
  uint32_t *qA = nullptr, *qH = nullptr, *qN = nullptr, *ctr = nullptr;  // cur/next, hit, NEE queues; counters
  uint32_t* hCtr = nullptr;  // page-locked copy of the counters
  void* spill = nullptr;     // traversal-stack spill area of the persistent kernels
  rt::Event evCtr;
  uint32_t capacity = 0;
  // A finished chunk leaves the lane at once: its per-path tail (the few paths that survive many bounces) and its
  // accumulate run on the lane's SIDE stream, on copies of the surviving paths' state (`ts`, same indexing as `ps`) and
  // on the chunk's own radiance buffer (two per lane), while the lane's stream starts the next chunk.
  rt::Stream side;
  PathState ts{};
  ShadowQueue tsq{};
  uint32_t* tq = nullptr;
  float4* Lbuf[2] = {nullptr, nullptr};
  int lSel = 0;
  bool accPending[2] = {false, false};  // Lbuf[b] holds a finished chunk whose accumulate is not launched yet
  rt::Event evChunk, evTail, evSide[2];  // end of the chunk's lane-stream work; tail buffers free; accumulate of Lbuf[b] done
  // chunk in flight
  bool active = false, waiting = false, done = false;
  uint32_t chunk = 0, n = 0, bounce = 0;
  WaveParams w{};
  uint32_t K = 0, sDone = 0;
};
constexpr uint32_t kTailCapacity = 65536;  // most paths a tail kernel takes over (YcOptions::tailThreshold is clamped to it)

struct yc_ctx {
  rt::Stream st;
  Lane lanes[kLanes];
  int device = 0, smCount = 1;
  std::string err;
  YcOptions opts{};
  uint32_t capacity = 0;

  std::vector<void*> sceneAllocs;
  DScene ds{};
  bool hasScene = false;
  YcCamera cam{};
  bool hasCamera = false;

  // frame
  bool inFrame = false;
  YcFrameDesc frame{};
  std::vector<uint32_t> pixels;  // this shard's pixels, tile-major: x | y << 16
  uint32_t* dPixels = nullptr;
  uint32_t* dPixelsScratch = nullptr;
  float4 *dHdr = nullptr, *dLdr = nullptr, *dBuckets = nullptr;
  size_t bucketCapacity = 0;  // pixels per bucket plane
  bool bucketsDirty = false;  // an accumulate was not (or only partly) followed by a finalize: the planes hold sums

  // wavefront storage lives in the lanes; the ray hooks (yc_trace*) use lane 0's counters and spill area
  uint32_t* dCtr = nullptr;
  void* dSpill = nullptr;
  Counters* dCounters = nullptr;
  std::vector<void*> waveAllocs;

  rt::Event ev0, ev1;
  // Waves issued by yc_render_wave_async and not yet waited for (every other entry point settles them first): the next
  // wave's chunks start while the previous wave's per-path tails, accumulates and finalize are still running.
  bool wavesPending = false;
  rt::Event evFinal;  // after the last finalize kernel: the bucket planes are zeroed, the next wave may accumulate
  std::vector<std::pair<rt::Event, rt::Event>> extendEvents;  // one pair per timed extend launch of the wave
  size_t extendEventsUsed = 0;
  std::vector<std::pair<rt::Event, rt::Event>> shadeEvents;   // the same for the surface-shading launches
  size_t shadeEventsUsed = 0;
  double shadeMs = 0, commMs = 0;
  uint64_t shadeLaunches = 0, hitsShaded = 0;
  bool timeShade = false;
  bool oneLane = false;  // profiling: chunks one after the other on lane 0, so that a launch's event time is its own
  uint64_t launches = 0;
  double gpuMs = 0, extendMs = 0;
  uint64_t extendLaunches = 0, raysExtend = 0;
  bool timeExtend = false, countTraversal = false;
  uint32_t tailThreshold = 16384;  // paths left in a chunk at which the tail kernel takes over (0 = never)
  const volatile int32_t* abortFlag = nullptr;  // yc_set_abort_flag
  std::unique_ptr<Comm> comm;      // yc_comm_*: the communicator this context belongs to
  bool wide = false;               // the scene's wide BVH is built and the kernels walk it (YcOptions::traversal)
  int wideDepth = 0;               // deepest wide level over all meshes
  uint64_t nWideNodes = 0;
};

static int settleWaves(yc_ctx* ctx);

static int fail(yc_ctx* c, int code, const char* fmt, ...) {
  if (c) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    c->err = buf;
  }
  return code;
}
#define YC_TRY(expr)                                                        \
  do {                                                                      \
    const char* e_ = (expr);                                                \
    if (e_) return fail(ctx, YC_ERR_CUDA, "%s: %s", #expr, e_);             \
  } while (0)

// Start of every entry point that touches the device: select it (the current device is per-thread state) and wait for
// waves still in flight from yc_render_wave_async — only that call and yc_comm_reduce_frames_async chain behind them.
static int enter(yc_ctx* ctx) {
  rt::useDevice(ctx->device);
  return ctx->wavesPending ? settleWaves(ctx) : YC_OK;
}
#define YC_ENTER(ctx)                        \
  do {                                       \
    if (const int e_ = enter(ctx)) return e_; \
  } while (0)

template <typename T>
static const char* devAlloc(std::vector<void*>& owner, T** p, size_t count) {
  void* v = nullptr;
  const char* e = rt::alloc(&v, count * sizeof(T));
  if (e) return e;
  owner.push_back(v);
  *p = static_cast<T*>(v);
  return nullptr;
}

template <typename T>
static const char* devUpload(yc_ctx* ctx, const T* src, size_t count, const T** out) {
  T* d = nullptr;
  const char* e = devAlloc(ctx->sceneAllocs, &d, count);
  if (e) return e;
  if (count && (e = rt::h2d(ctx->st, d, src, count * sizeof(T)))) return e;
  *out = d;
  return nullptr;
}

static void freeAll(std::vector<void*>& v) {
  for (void* p : v) rt::release(p);
  v.clear();
}

// ---------------------------------------------------------------------------------------
// stages as functors (run by rt::launchFor) and the two persistent traversal kernels
// ---------------------------------------------------------------------------------------
struct RaygenK {
  WaveParams w;
  PathState ps;
  uint32_t* queue;
  YB_DEV void operator()(uint32_t i) const {
    raygenStage(w, ps, i);
    queue[i] = i;
  }
};

// Surface shading over the HIT queue extend produced (count on the device: the launches are sized for the upper
// bound and surplus threads leave at once), in three kernels (integrator.cuh: resolveSurface / sampleSurface /
// shadeNee): the first gathers each hit's surface into a SurfRecord at the hit's queue position, the second samples
// the BSDF from it and appends the surviving paths to the next queue and the hits that take a NEE sample to the NEE
// queue, the third turns those into shadow requests.
struct ResolveK {
  DScene sc;
  PathState ps;
  SurfState ss;
  const uint32_t* queue;
  const uint32_t* ctr;
  YB_DEV void operator()(uint32_t j) const {
    if (j >= ctr[kCtrHitCount]) return;
    storeSurf(ss, j, resolveSurface(sc, ps, queue[j]));
  }
};

template <bool DEFER_RR>
struct SampleK {
  DScene sc;
  WaveParams w;
  PathState ps;
  SurfState ss;
  const uint32_t* queue;
  uint32_t *nextQueue, *neeQueue;
  uint32_t* ctr;
  Counters* counters;
  YB_DEV void operator()(uint32_t j) const {
    if (j >= ctr[kCtrHitCount]) return;
    const uint32_t i = queue[j];
    V3 neeAtt;
    uint32_t neeDim = 0, rays = 0;
    const uint32_t r = sampleSurface<DEFER_RR>(sc, w, ps, i, loadSurf(ss, j), neeAtt, neeDim, rays);
    aggregatedCount(&counters->raysReference, rays);
    if (r & kShadeContinue) nextQueue[aggregatedAppend(ctr + kCtrNextCount)] = i;
    if (r & kShadeNee) {
      ss.r7[j] = make_float4(neeAtt.x, neeAtt.y, neeAtt.z, __uint_as_float(neeDim));
      neeQueue[aggregatedAppend(ctr + kCtrNeeCount)] = j;
    }
  }
};

struct ShadeNeeK {
  DScene sc;
  WaveParams w;
  SurfState ss;
  ShadowQueue sq;
  const uint32_t *queue, *neeQueue;  // hit queue (position → path), NEE queue (positions in the hit queue)
  uint32_t* ctr;
  YB_DEV void operator()(uint32_t k) const {
    if (k >= ctr[kCtrNeeCount]) return;
    const uint32_t j = neeQueue[k];
    const uint32_t i = queue[j];
    const float4 x = ss.r7[j];
    ShadowRequest rq;
    if (shadeNee(sc, w, i, loadSurf(ss, j), V3(x.x, x.y, x.z), __float_as_uint(x.w), rq)) {
      const uint32_t q = aggregatedAppend(ctr + kCtrShadowCount);
      sq.o[q] = make_float4(rq.o.x, rq.o.y, rq.o.z, rq.tMax);
      sq.d[q] = make_float4(rq.d.x, rq.d.y, rq.d.z, rq.absDotN);
      sq.lif[q] = make_float4(rq.lif.x, rq.lif.y, rq.lif.z, rq.denom);
      sq.att[q] = make_float4(rq.att.x, rq.att.y, rq.att.z, __uint_as_float(i));
    }
  }
};

// After extend: the bounce's hits go to the hit queue (one warp-aggregated append per warp, so that the heavy surface
// shading runs in full warps; appending from inside the persistent extend kernel costs one atomic per ray), its misses
// are shaded on the spot — environment lights with their MIS weight, background (mis-integrator.cpp:27-43): a few
// texel taps, not worth a queue and a launch of their own — and paths killed by a deferred roulette drop out.
struct SortMissK {
  DScene sc;
  WaveParams w;
  PathState ps;
  const uint32_t* queue;
  uint32_t *hitQueue, *ctr;
  Counters* counters;
  YB_DEV void operator()(uint32_t j) const {
    const uint32_t i = queue[j];
    const int32_t hb = ps.hitB[i];
    uint32_t rays = 0;
    if (hb >= 0) hitQueue[aggregatedAppend(ctr + kCtrHitCount)] = i;
    else if (hb == kHitMiss) shadeMissStage(sc, w, ps, i, rays);
    aggregatedCount(&counters->raysReference, rays);  // (per group of lanes, if the branches above have not reconverged)
  }
};

// Integrator::render's estimator.addSample loop for one chunk (integrator.cpp:19-24): pixel p adds
// its K samples in sample order into bucket (sample index within the wave) % m.
struct AccumulateK {
  PathState ps;
  float4* buckets;
  size_t planeStride;
  uint32_t pixBase, nPix, K, waveSampleBase, sampleStride, m, estimator;
  float exposureScale;
  YB_DEV void operator()(uint32_t p) const {
    for (uint32_t k = 0; k < K; k++) {
      const float4 L4 = ps.L[size_t(k) * nPix + p];
      const V3 s = V3(L4.x, L4.y, L4.z) * exposureScale;
      const uint32_t b = estimator == YC_ESTIMATOR_MEAN ? 0u : (waveSampleBase + k * sampleStride) % m;
      if (estimatorAccepts(int(estimator), s)) {
        float4* slot = buckets + size_t(b) * planeStride + (pixBase + p);
        float4 v = *slot;
        v.x += s.x, v.y += s.y, v.z += s.z;
        v.w = __uint_as_float(__float_as_uint(v.w) + 1u);
        *slot = v;
      }
    }
  }
};

// Estimator::getValue + TileRenderer::finishTile's blend and tonemap (tile-renderer.hpp:220-239).
struct FinalizeK {
  const uint32_t* pixelList;
  float4* buckets;
  size_t planeStride;
  float4 *hdr, *ldr;
  float4 *hdrRoot, *ldrRoot;  // tile sharding over GPUs that reach the root's memory (comm.cuh): the combined frames, else null
  uint32_t width, m, estimator, waveSamples, tonemap;
  float wCurrent, wWave;
  YB_DEV void operator()(uint32_t p) const {
    V3 acc[kMaxBuckets];
    uint32_t cnt[kMaxBuckets];
    for (uint32_t b = 0; b < m; b++) {
      float4* slot = buckets + size_t(b) * planeStride + p;
      const float4 v = *slot;
      acc[b] = V3(v.x, v.y, v.z);
      cnt[b] = __float_as_uint(v.w);
      *slot = make_float4(0.0f, 0.0f, 0.0f, 0.0f);  // ready for the next wave
    }
    const V3 wave = estimatorValue(int(estimator), acc, cnt, int(m), waveSamples);
    const uint32_t pix = pixelList[p];
    const size_t idx = size_t(pix >> 16) * width + (pix & 0xffffu);
    const float4 cur = hdr[idx];
    float4 h;
    h.x = cur.x * wCurrent + wave.x * wWave;
    h.y = cur.y * wCurrent + wave.y * wWave;
    h.z = cur.z * wCurrent + wave.z * wWave;
    h.w = cur.w * wCurrent + 1.0f * wWave;
    hdr[idx] = h;
    float4 l = h;
    if (tonemap != YC_TONEMAP_NONE) {
      const V3 t = agx(V3(h.x, h.y, h.z), agxLook(tonemap));
      l = make_float4(t.x, t.y, t.z, 1.0f);
    }
    ldr[idx] = l;
    if (hdrRoot) hdrRoot[idx] = h, ldrRoot[idx] = l;  // stores over NVLink when the root is another GPU
  }
};

// Tile sharding, direct delivery: this shard's pixels of the own frames into the root's combined frames (the first
// wave after the frames were mapped, or after a wave that finalized only part of the shard).
struct PushFramesK {
  const uint32_t* pixelList;
  const float4 *hdr, *ldr;
  float4 *hdrRoot, *ldrRoot;
  uint32_t width;
  YB_DEV void operator()(uint32_t p) const {
    const uint32_t pix = pixelList[p];
    const size_t idx = size_t(pix >> 16) * width + (pix & 0xffffu);
    hdrRoot[idx] = hdr[idx], ldrRoot[idx] = ldr[idx];
  }
};

struct RetonemapK {
  float4 *hdr, *ldr;
  uint32_t tonemap;
  YB_DEV void operator()(uint32_t idx) const {
    const float4 h = hdr[idx];
    if (tonemap == YC_TONEMAP_NONE) {
      ldr[idx] = h;
    } else {
      const V3 t = agx(V3(h.x, h.y, h.z), agxLook(tonemap));
      ldr[idx] = make_float4(t.x, t.y, t.z, 1.0f);
    }
  }
};

#ifdef YB_HOSTSIM
struct HostStack {
  uint32_t ref[kShStack];
  float d[kShStack];
  TravStack ts;
  HostStack() {
    ts.shRef = ref;
    ts.shD = d;
    ts.stride = 1;
  }
};
template <bool ALPHA, bool COUNT>
static void runExtend(yc_ctx* ctx, Lane& L, uint32_t n) {
  HostStack hs;
  TraceCounters cnt;
  if (!ALPHA && ctx->wide && !COUNT)
    for (uint32_t j = 0; j < n; j++) extendStage<false, false, WideWalk>(ctx->ds, L.w, L.ps, L.qA[j], hs.ts, cnt);
  else
    for (uint32_t j = 0; j < n; j++) extendStage<ALPHA, COUNT, Bvh2Walk>(ctx->ds, L.w, L.ps, L.qA[j], hs.ts, cnt);
  ctx->dCounters->boxTests += cnt.box;
  ctx->dCounters->triTests += cnt.tri;
}
template <bool ALPHA, bool COUNT>
static void runShadow(yc_ctx* ctx, Lane& L, uint32_t) {
  HostStack hs;
  TraceCounters cnt;
  const uint32_t n = L.ctr[kCtrShadowCount];
  uint32_t contributed = 0;
  if (!ALPHA && ctx->wide && !COUNT)
    for (uint32_t j = 0; j < n; j++) contributed += shadowStage<false, false, WideWalk>(ctx->ds, L.w, L.ps, L.sq, j, hs.ts, cnt);
  else
    for (uint32_t j = 0; j < n; j++) contributed += shadowStage<ALPHA, COUNT, Bvh2Walk>(ctx->ds, L.w, L.ps, L.sq, j, hs.ts, cnt);
  ctx->dCounters->raysShadow += n;
  ctx->dCounters->raysReference += contributed;
  ctx->dCounters->boxTests += cnt.box;
  ctx->dCounters->triTests += cnt.tri;
}
template <bool ALPHA>
static void runNaive(yc_ctx* ctx, Lane& L) {
  HostStack hs;
  TraceCounters cnt;
  uint32_t rays = 0;
  for (uint32_t j = 0; j < L.n; j++) naiveStage<ALPHA>(ctx->ds, L.w, L.ps, L.qA[j], hs.ts, cnt, rays);
  ctx->dCounters->raysReference += rays;
  ctx->dCounters->raysExtend += rays;
}
#else
// Persistent extend / shadow kernels: IO adapters around tracePersistent (trace_kernels.cuh), one kernel per BVH
// layout; the wide ones serve scenes without alpha-tested materials.
#ifndef YB_WIDE_MIN_BLOCKS
#define YB_WIDE_MIN_BLOCKS 7  // 72 registers, no spills (6 CTAs: 80 registers, soup trace 3.32 ms; 7: 3.10 ms; 8 spills: 3.24 ms)
#endif

// Counting builds add their box and triangle tests to `counters`.
template <bool COUNT>
__device__ __forceinline__ void flushCounts(Counters* counters, const TraceCounters& cnt) {
  if (COUNT) {
    aggregatedCount(&counters->boxTests, cnt.box);
    aggregatedCount(&counters->triTests, cnt.tri);
  }
}

template <bool ALPHA>
struct ExtendIO {
  WaveParams w;
  PathState ps;
  const uint32_t* queue;
  __device__ __forceinline__ bool load(uint32_t j, V3& o, V3& d, float& tMax, Sampler& smp) const {
    tMax = INFINITY;
    return extendLoad<ALPHA>(w, ps, queue[j], o, d, smp);
  }
  __device__ __forceinline__ void store(uint32_t j, const TraceState& st, bool, const Sampler& smp) const {
    extendStore<ALPHA>(ps, queue[j], st, smp);
  }
};

template <bool ALPHA, bool COUNT>
__global__ void __launch_bounds__(kTraceBlock, YB_TRACE_MIN_BLOCKS) extendKernel(DScene sc, WaveParams w, PathState ps, const uint32_t* queue,
                                                            uint32_t n, uint32_t* ctr, Counters* counters, uint2* spill,
                                                            TraceTuning tune) {
  ExtendIO<ALPHA> io{w, ps, queue};
  TraceCounters cnt;
  tracePersistent<Bvh2Walk, false, ALPHA, COUNT, false>(sc, io, n, ctr + kCtrExtendHead, spill, tune, cnt);
  flushCounts<COUNT>(counters, cnt);
}
__global__ void __launch_bounds__(kTraceBlock, YB_WIDE_MIN_BLOCKS) extendWideKernel(DScene sc, WaveParams w, PathState ps, const uint32_t* queue,
                                                              uint32_t n, uint32_t* ctr, Counters* counters, uint2* spill,
                                                              TraceTuning tune) {
  ExtendIO<false> io{w, ps, queue};
  TraceCounters cnt;
  tracePersistent<WideWalk, false, false, false, false>(sc, io, n, ctr + kCtrExtendHead, spill, tune, cnt);
}

template <bool ALPHA>
struct ShadowIO {
  WaveParams w;
  PathState ps;
  ShadowQueue sq;
  uint32_t contributed = 0;
  uint32_t pathOf[1];  // unused
  __device__ __forceinline__ bool load(uint32_t j, V3& o, V3& d, float& tMax, Sampler& smp) const {
    shadowLoad<ALPHA>(w, ps, sq, j, o, d, tMax, smp);
    return true;
  }
  __device__ __forceinline__ void store(uint32_t j, const TraceState& st, bool occluded, const Sampler& smp) {
    contributed += shadowFinish<ALPHA>(ps, sq, j, __float_as_uint(sq.att[j].w), st, occluded, smp);
  }
};

// EARLY_OUT = !ALPHA: see shadowStage (integrator.cuh)
template <class Walk, bool ALPHA, bool COUNT>
__device__ __forceinline__ void shadowQueue(const DScene& sc, WaveParams w, PathState ps, ShadowQueue sq, uint32_t* ctr, Counters* counters,
                                            uint2* spill, const TraceTuning& tune) {
  const uint32_t n = ctr[kCtrShadowCount];
  ShadowIO<ALPHA> io{w, ps, sq};
  TraceCounters cnt;
  tracePersistent<Walk, true, ALPHA, COUNT, !ALPHA>(sc, io, n, ctr + kCtrShadowHead, spill, tune, cnt);
  aggregatedCount(&counters->raysReference, io.contributed);
  if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(&counters->raysShadow, (unsigned long long)n);
  flushCounts<COUNT>(counters, cnt);
}
template <bool ALPHA, bool COUNT>
__global__ void __launch_bounds__(kTraceBlock, YB_SHADOW_MIN_BLOCKS) shadowKernel(DScene sc, WaveParams w, PathState ps, ShadowQueue sq,
                                                            uint32_t* ctr, Counters* counters, uint2* spill, TraceTuning tune) {
  shadowQueue<Bvh2Walk, ALPHA, COUNT>(sc, w, ps, sq, ctr, counters, spill, tune);
}
__global__ void __launch_bounds__(kTraceBlock, YB_WIDE_MIN_BLOCKS) shadowWideKernel(DScene sc, WaveParams w, PathState ps, ShadowQueue sq,
                                                              uint32_t* ctr, Counters* counters, uint2* spill, TraceTuning tune) {
  shadowQueue<WideWalk, false, false>(sc, w, ps, sq, ctr, counters, spill, tune);
}

// Tail of a chunk: once only a few thousand paths survive, every further bounce of the wavefront is
// bound by the latency of its slowest ray (launch after launch).  The tail kernel gives each surviving
// path one thread that runs its remaining bounces to the end — extend → shade → shadow in the same
// order and with the same stage functions as the wavefront, so results are unchanged — and all the
// slow rays overlap instead of adding up.
constexpr int kTailBlock = 128;
// The surviving paths' state copied out of the lane's arrays (same index), so that the lane can start its next chunk.
struct TailGatherK {
  PathState ps, ts;
  const uint32_t* queue;
  uint32_t* tq;
  YB_DEV void operator()(uint32_t j) const {
    const uint32_t i = queue[j];
    tq[j] = i;
    ts.rayO[i] = ps.rayO[i], ts.rayD[i] = ps.rayD[i], ts.L[i] = ps.L[i], ts.att[i] = ps.att[i];
    ts.dim[i] = ps.dim[i], ts.flags[i] = ps.flags[i];
  }
};

template <bool ALPHA, class Walk>
__global__ void __launch_bounds__(kTailBlock) tailKernel(DScene sc, WaveParams w, PathState ps, ShadowQueue sq,
                                                         const uint32_t* queue, uint32_t n, uint32_t firstBounce,
                                                         Counters* counters, float4* Lout) {
  __shared__ uint32_t shRef[kShStack * kTailBlock];
  __shared__ float shD[kShStack * kTailBlock];
  TravStack stack;
  stack.shRef = shRef + threadIdx.x;
  stack.shD = shD + threadIdx.x;
  stack.stride = kTailBlock;
  const uint32_t j = blockIdx.x * kTailBlock + threadIdx.x;
  uint32_t raysRef = 0, nExtend = 0, nShadow = 0;
  if (j < n) {
    const uint32_t i = queue[j];
    TraceCounters cnt;
    for (uint32_t bounce = firstBounce; bounce < w.maxDepth; bounce++) {
      extendStage<ALPHA, false, Walk>(sc, w, ps, i, stack, cnt);
      nExtend++;
      ShadowRequest rq;
      const uint32_t r = shadeStage<ALPHA>(sc, w, ps, i, rq, raysRef);
      if (r & kShadeShadow) {
        // slot j of the NEE queue is this thread's own
        sq.o[j] = make_float4(rq.o.x, rq.o.y, rq.o.z, rq.tMax);
        sq.d[j] = make_float4(rq.d.x, rq.d.y, rq.d.z, rq.absDotN);
        sq.lif[j] = make_float4(rq.lif.x, rq.lif.y, rq.lif.z, rq.denom);
        sq.att[j] = make_float4(rq.att.x, rq.att.y, rq.att.z, __uint_as_float(i));
        raysRef += shadowStage<ALPHA, false, Walk>(sc, w, ps, sq, j, stack, cnt);
        nShadow++;
      }
      if (!(r & kShadeContinue)) break;
    }
    Lout[i] = ps.L[i];  // back into the chunk's radiance buffer, where the accumulate reads it
  }
  __syncwarp();
  aggregatedCount(&counters->raysReference, raysRef);
  aggregatedCount(&counters->raysExtend, nExtend);
  aggregatedCount(&counters->raysShadow, nShadow);
}

// NaiveIntegrator: one thread per path, whole path (integrator.cuh naiveStage).
template <bool ALPHA>
__global__ void __launch_bounds__(kTailBlock) naiveKernel(DScene sc, WaveParams w, PathState ps, const uint32_t* queue, uint32_t n,
                                                          Counters* counters) {
  __shared__ uint32_t shRef[kShStack * kTailBlock];
  __shared__ float shD[kShStack * kTailBlock];
  TravStack stack;
  stack.shRef = shRef + threadIdx.x;
  stack.shD = shD + threadIdx.x;
  stack.stride = kTailBlock;
  const uint32_t j = blockIdx.x * kTailBlock + threadIdx.x;
  uint32_t rays = 0;
  if (j < n) {
    TraceCounters cnt;
    naiveStage<ALPHA>(sc, w, ps, queue[j], stack, cnt, rays);
  }
  __syncwarp();
  aggregatedCount(&counters->raysReference, rays);
  aggregatedCount(&counters->raysExtend, rays);
}
template <bool ALPHA>
static void runNaive(yc_ctx* ctx, Lane& L) {
  naiveKernel<ALPHA><<<(L.n + kTailBlock - 1) / kTailBlock, kTailBlock, 0, L.st.s>>>(ctx->ds, L.w, L.ps, L.qA, L.n, ctx->dCounters);
}

static int traceGridMax(const yc_ctx* ctx) { return ctx->smCount * 8; }
static TraceTuning tuning(const yc_ctx* ctx) {
  TraceTuning t;
  t.refillMin = ctx->opts.traceRefillMin ? int(ctx->opts.traceRefillMin) : 8;
  t.innerMin = ctx->opts.traceInnerMin ? int(ctx->opts.traceInnerMin) : 20;
  const int e = ctx->opts.sharedStackEntries ? int(ctx->opts.sharedStackEntries) : kPsStack;
  t.shEntries = std::max(2, std::min(kPsStack, e));
  return t;
}
static int traceGrid(const yc_ctx* ctx, uint32_t n) {
  // persistent: enough CTAs to fill every SM (registers / shared memory cap residency below this)
  const int needed = int((n + kTraceBlock - 1) / kTraceBlock);
  return std::max(1, std::min(traceGridMax(ctx), needed));
}

template <bool ALPHA, bool COUNT>
static void runExtend(yc_ctx* ctx, Lane& L, uint32_t n) {
  std::pair<rt::Event, rt::Event>* ev = nullptr;
  if (ctx->timeExtend) {
    if (ctx->extendEventsUsed == ctx->extendEvents.size()) {
      ctx->extendEvents.emplace_back();
      rt::eventCreate(ctx->extendEvents.back().first);
      rt::eventCreate(ctx->extendEvents.back().second);
    }
    ev = &ctx->extendEvents[ctx->extendEventsUsed++];
    rt::eventRecord(L.st, ev->first);
  }
  const auto kernel = !ALPHA && !COUNT && ctx->wide ? extendWideKernel : extendKernel<ALPHA, COUNT>;
  kernel<<<traceGrid(ctx, n), kTraceBlock, 0, L.st.s>>>(ctx->ds, L.w, L.ps, L.qA, n, L.ctr, ctx->dCounters, static_cast<uint2*>(L.spill),
                                                       tuning(ctx));
  if (ev) rt::eventRecord(L.st, ev->second);
}
template <bool ALPHA, bool COUNT>
static void runShadow(yc_ctx* ctx, Lane& L, uint32_t upperBound) {
  const auto kernel = !ALPHA && !COUNT && ctx->wide ? shadowWideKernel : shadowKernel<ALPHA, COUNT>;
  kernel<<<traceGrid(ctx, upperBound), kTraceBlock, 0, L.st.s>>>(ctx->ds, L.w, L.ps, L.sq, L.ctr, ctx->dCounters,
                                                                static_cast<uint2*>(L.spill), tuning(ctx));
}
#endif

// ---------------------------------------------------------------------------------------
// lifecycle
// ---------------------------------------------------------------------------------------
extern "C" int yc_create(int device, const YcOptions* opts, yc_ctx** out) {
  if (!out) return YC_ERR_INVALID;
  *out = nullptr;
  yc_ctx* ctx = new (std::nothrow) yc_ctx();
  if (!ctx) return YC_ERR_INVALID;
  if (opts) ctx->opts = *opts;
  if (ctx->opts.maxDepth == 0) ctx->opts.maxDepth = 30;  // RayIntegrator::m_maxDepth, ray-integrator.hpp:14
  if (ctx->opts.integrator > YC_INTEGRATOR_NAIVE || ctx->opts.scrambler > YC_SCRAMBLER_BINARY_PERMUTE ||
      ctx->opts.sampler > YC_SAMPLER_STRATIFIED || ctx->opts.lightSampler > YC_LIGHT_SAMPLER_UNIFORM ||
      ctx->opts.traversal > YC_TRAVERSAL_WIDE ||
      (ctx->opts.integrator == YC_INTEGRATOR_NAIVE && ctx->opts.maxDepth + 1 > kNaiveMaxSegments)) {
    delete ctx;
    return YC_ERR_INVALID;
  }
#ifndef YB_RNG_SAMPLERS
  if (ctx->opts.sampler != YC_SAMPLER_SOBOL || ctx->opts.scrambler != YC_SCRAMBLER_FAST_OWEN ||
      ctx->opts.lightSampler != YC_LIGHT_SAMPLER_POWER) {
    // this build folds the sampler choice away (sampler.cuh); the other samplers are in libyart_b200_samplers.so
    delete ctx;
    return YC_ERR_UNSUPPORTED;
  }
#endif
  ctx->capacity = ctx->opts.maxPathsInFlight ? ctx->opts.maxPathsInFlight : (8u << 20);
  if (ctx->opts.tailThreshold) ctx->tailThreshold = ctx->opts.tailThreshold == 0xffffffffu ? 0u : ctx->opts.tailThreshold;
  ctx->device = device;
  const char* e = rt::init(device, ctx->st, ctx->smCount);
  if (e) {
    // there is no CPU fallback: without a usable device the context does not exist
    fprintf(stderr, "yart_b200: cannot create a CUDA context on device %d: %s\n", device, e);
    delete ctx;
    return YC_ERR_NO_DEVICE;
  }
  rt::eventCreate(ctx->ev0);
  rt::eventCreate(ctx->ev1);
  rt::eventCreate(ctx->evFinal);
  for (int l = 0; l < kLanes; l++) {
    Lane& L = ctx->lanes[l];
    if (const char* le = rt::streamCreate(L.st)) {
      fprintf(stderr, "yart_b200: cannot create a stream: %s\n", le);
      delete ctx;
      return YC_ERR_CUDA;
    }
    if (const char* le = rt::streamCreate(L.side)) {
      fprintf(stderr, "yart_b200: cannot create a stream: %s\n", le);
      delete ctx;
      return YC_ERR_CUDA;
    }
    rt::eventCreate(L.evCtr);
    rt::eventCreate(L.evChunk);
    rt::eventCreate(L.evTail);
    rt::eventCreate(L.evSide[0]);
    rt::eventCreate(L.evSide[1]);
  }
  if (ctx->tailThreshold > kTailCapacity) ctx->tailThreshold = kTailCapacity;
  *out = ctx;
  return YC_OK;
}

static void freeFrame(yc_ctx* ctx) {
  rt::release(ctx->dPixels);
  rt::release(ctx->dPixelsScratch);
  rt::release(ctx->dHdr);
  rt::release(ctx->dLdr);
  rt::release(ctx->dBuckets);
  ctx->dPixels = ctx->dPixelsScratch = nullptr;
  ctx->dHdr = ctx->dLdr = ctx->dBuckets = nullptr;
  ctx->inFrame = false;
}

static void destroyComm(yc_ctx* ctx);
static void detachCombinedFrames(yc_ctx* ctx);

extern "C" void yc_destroy(yc_ctx* ctx) {
  if (!ctx) return;
  enter(ctx);
  rt::sync(ctx->st);
  destroyComm(ctx);
  freeFrame(ctx);
  freeAll(ctx->sceneAllocs);
  freeAll(ctx->waveAllocs);
  rt::eventDestroy(ctx->ev0);
  rt::eventDestroy(ctx->ev1);
  rt::eventDestroy(ctx->evFinal);
  for (auto* evs : {&ctx->extendEvents, &ctx->shadeEvents})
    for (auto& ev : *evs) {
      rt::eventDestroy(ev.first);
      rt::eventDestroy(ev.second);
    }
  for (int l = 0; l < kLanes; l++) {
    Lane& L = ctx->lanes[l];
    rt::sync(L.st);
    rt::sync(L.side);
    rt::hostRelease(L.hCtr);
    rt::eventDestroy(L.evCtr);
    rt::eventDestroy(L.evChunk);
    rt::eventDestroy(L.evTail);
    rt::eventDestroy(L.evSide[0]);
    rt::eventDestroy(L.evSide[1]);
    rt::destroy(L.side);
    rt::destroy(L.st);
  }
  rt::destroy(ctx->st);
  delete ctx;
}

extern "C" const char* yc_last_error(const yc_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }

extern "C" int yc_synchronize(yc_ctx* ctx) {
  if (!ctx) return YC_ERR_INVALID;
  YC_ENTER(ctx);
  YC_TRY(rt::sync(ctx->st));
  return YC_OK;
}

extern "C" int yc_upload_scene(yc_ctx* ctx, const YcScene* s) {
  if (!ctx || !s) return YC_ERR_INVALID;
  YC_ENTER(ctx);
  if (!s->nodes || s->nNodes == 0 || !s->lutTables) return fail(ctx, YC_ERR_INVALID, "scene has no nodes or no LUT tables");
  for (uint32_t i = 0; i < s->nNodes; i++) {
    const YcNode& n = s->nodes[i];
    if (n.depth < 0 || n.depth >= YC_MAX_NODE_DEPTH || n.skip <= int32_t(i) || n.skip > int32_t(s->nNodes) ||
        n.mesh >= int32_t(s->nMeshes) || n.parent >= int32_t(i) || (i == 0) != (n.parent < 0) ||
        (n.parent >= 0 && n.depth != s->nodes[n.parent].depth + 1) || (n.parent < 0 && n.depth != 0))
      return fail(ctx, YC_ERR_INVALID, "node %u is inconsistent (depth/skip/mesh/parent)", i);
  }
  for (uint64_t i = 0; i < s->nPrims; i++)
    if (s->primMaterial[i] >= s->nMaterials) return fail(ctx, YC_ERR_INVALID, "primitive %llu: bad material", (unsigned long long)i);
  // The traversal stack holds at most one entry per level (testBVH pushes the far child and descends into the near
  // one), the reference's is `stack[64]` (ray-integrator.cpp:92-93) and overflows silently beyond that; here a
  // deeper tree is refused instead of walking off the spill area.
  for (uint32_t mi = 0; mi < s->nMeshes; mi++) {
    const YcMesh& m = s->meshes[mi];
    if (uint64_t(m.nodeOffset) + m.nInner > s->nBvhNodes) return fail(ctx, YC_ERR_INVALID, "mesh %u: BVH nodes out of range", mi);
    if (m.rootRef & YC_REF_LEAF) continue;
    std::vector<std::pair<uint32_t, int>> todo{{m.rootRef, 1}};
    size_t visited = 0;
    while (!todo.empty()) {
      const auto [ref, depth] = todo.back();
      todo.pop_back();
      if (ref >= m.nInner || ++visited > m.nInner) return fail(ctx, YC_ERR_INVALID, "mesh %u: BVH is not a tree", mi);
      if (depth > kMaxStack) return fail(ctx, YC_ERR_INVALID, "mesh %u: BVH deeper than %d levels", mi, kMaxStack);
      const YcBvhNode& n = s->bvhNodes[size_t(m.nodeOffset) + ref];
      if (!(n.ref0 & YC_REF_LEAF)) todo.push_back({n.ref0, depth + 1});
      if (!(n.ref1 & YC_REF_LEAF)) todo.push_back({n.ref1, depth + 1});
    }
  }
  YC_TRY(rt::sync(ctx->st));
  freeAll(ctx->sceneAllocs);
  ctx->hasScene = false;
  DScene d{};
  const YcBvhNode* bn = nullptr;
  const YcBvhTri* bt = nullptr;
  YC_TRY(devUpload(ctx, s->nodes, s->nNodes, &d.nodes));
  {
    std::vector<int32_t> path(size_t(s->nNodes) * YC_MAX_NODE_DEPTH, 0);
    for (uint32_t i = 0; i < s->nNodes; i++) {
      int32_t a = int32_t(i);
      for (int level = s->nodes[i].depth; level >= 0 && a >= 0; level--) {
        path[size_t(i) * YC_MAX_NODE_DEPTH + level] = a;
        a = s->nodes[a].parent;
      }
    }
    YC_TRY(devUpload(ctx, path.data(), path.size(), &d.nodePath));
  }
  YC_TRY(devUpload(ctx, s->meshes, s->nMeshes, &d.meshes));
  YC_TRY(devUpload(ctx, s->bvhNodes, size_t(s->nBvhNodes), &bn));
  YC_TRY(devUpload(ctx, s->bvhTris, size_t(s->nBvhTris), &bt));
  d.bvhNodes = reinterpret_cast<const float4*>(bn);
  d.bvhTris = reinterpret_cast<const float4*>(bt);
  // the wide (4-ary) layout of the same trees (wide_bvh.cuh), for scenes whose triangle-test order cannot move
  // sampler draws; a wide walk pushes up to three entries per level
  ctx->wide = false, ctx->wideDepth = 0, ctx->nWideNodes = 0;
  if (ctx->opts.traversal == YC_TRAVERSAL_WIDE && s->hasAlpha)
    return fail(ctx, YC_ERR_UNSUPPORTED, "YC_TRAVERSAL_WIDE: the scene has alpha-tested materials");
  if (ctx->opts.traversal != YC_TRAVERSAL_REFERENCE_ORDER && !s->hasAlpha && s->nMeshes) {
    std::vector<WideNode> wn;
    std::vector<WideMesh> wm(s->nMeshes);
    int depth = 0;
    bool quantised = true;  // every mesh's boxes fit the quantised grid (quantiseWideNode)
    for (uint32_t mi = 0; mi < s->nMeshes; mi++) {
      const int dm = collapseToWide(s->bvhNodes + s->meshes[mi].nodeOffset, s->meshes[mi], wn, wm[mi]);
      quantised = quantised && dm >= 0;
      depth = std::max(depth, dm);
    }
    if (!quantised) {
      if (ctx->opts.traversal == YC_TRAVERSAL_WIDE)
        return fail(ctx, YC_ERR_UNSUPPORTED, "YC_TRAVERSAL_WIDE: a mesh's extent does not fit the wide nodes' quantised grid");
    } else if (3 * depth <= kMaxStack) {
      const WideNode* dw = nullptr;
      if (wn.empty()) wn.emplace_back();
      YC_TRY(devUpload(ctx, wn.data(), wn.size(), &dw));
      YC_TRY(devUpload(ctx, wm.data(), wm.size(), &d.wideMeshes));
      d.wideNodes = reinterpret_cast<const float4*>(dw);
      ctx->wide = true, ctx->wideDepth = depth, ctx->nWideNodes = wn.size();
    } else if (ctx->opts.traversal == YC_TRAVERSAL_WIDE) {
      return fail(ctx, YC_ERR_UNSUPPORTED, "YC_TRAVERSAL_WIDE: wide tree of %d levels exceeds the traversal stack", depth);
    }
  }
  YC_TRY(devUpload(ctx, s->positions, size_t(s->nVerts) * 3, &d.positions));
  YC_TRY(devUpload(ctx, s->normals, size_t(s->nVerts) * 3, &d.normals));
  YC_TRY(devUpload(ctx, s->tangents, size_t(s->nVerts) * 4, &d.tangents));
  YC_TRY(devUpload(ctx, s->uvs, size_t(s->nVerts) * 2, &d.uvs));
  YC_TRY(devUpload(ctx, s->primIndices, size_t(s->nPrims) * 3, &d.primIndices));
  YC_TRY(devUpload(ctx, s->primMaterial, size_t(s->nPrims), &d.primMaterial));
  YC_TRY(devUpload(ctx, s->primLight, size_t(s->nPrims), &d.primLight));
  YC_TRY(devUpload(ctx, s->materials, s->nMaterials, &d.materials));
  YC_TRY(devUpload(ctx, s->textures, s->nTextures, &d.textures));
  YC_TRY(devUpload(ctx, s->texelsU8, size_t(s->nTexelsU8), &d.texU8));
  YC_TRY(devUpload(ctx, s->texelsF32, size_t(s->nTexelsF32), &d.texF32));
  YC_TRY(devUpload(ctx, s->lights, s->nLights, &d.lights));
  YC_TRY(devUpload(ctx, s->envDist, size_t(s->nEnvDist), &d.envDist));
  YC_TRY(devUpload(ctx, s->infiniteLights, s->nInfinite, &d.infLights));
  YC_TRY(devUpload(ctx, s->areaLights, s->nArea, &d.areaLights));
  YC_TRY(devUpload(ctx, s->lightPowerCdf, s->nArea, &d.powerCdf));
  YC_TRY(devUpload(ctx, s->lutTables, 14112, &d.lut));
  d.nNodes = s->nNodes, d.nMeshes = s->nMeshes, d.nLights = s->nLights;
  d.nInf = s->nInfinite, d.nArea = s->nArea, d.totalPower = s->totalPower, d.hasAlpha = s->hasAlpha;
  d.uniformLights = ctx->opts.lightSampler == YC_LIGHT_SAMPLER_UNIFORM ? 1u : 0u;
  ctx->ds = d;
  ctx->hasScene = true;
  return YC_OK;
}

extern "C" int yc_set_camera(yc_ctx* ctx, const YcCamera* cam) {
  if (!ctx || !cam) return YC_ERR_INVALID;
  YC_ENTER(ctx);
  ctx->cam = *cam;
  ctx->hasCamera = true;
  return YC_OK;
}

static int ensureWaveStorage(yc_ctx* ctx) {
  if (!ctx->waveAllocs.empty()) return YC_OK;
  auto& own = ctx->waveAllocs;
  for (int l = 0; l < kLanes; l++) {
    Lane& L = ctx->lanes[l];
    L.capacity = std::max<uint32_t>(1u, ctx->capacity / kLanes);
    const size_t P = L.capacity;
    YC_TRY(devAlloc(own, &L.ps.rayO, P));
    YC_TRY(devAlloc(own, &L.ps.rayD, P));
    YC_TRY(devAlloc(own, &L.Lbuf[0], P));
    YC_TRY(devAlloc(own, &L.Lbuf[1], P));
    L.ps.L = L.Lbuf[0];
    YC_TRY(devAlloc(own, &L.ps.att, P));
    YC_TRY(devAlloc(own, &L.ps.dim, P));
    YC_TRY(devAlloc(own, &L.ps.flags, P));
    YC_TRY(devAlloc(own, &L.ps.hitA, P));
    YC_TRY(devAlloc(own, &L.ps.hitB, P));
    YC_TRY(devAlloc(own, &L.sq.o, P));
    YC_TRY(devAlloc(own, &L.sq.d, P));
    YC_TRY(devAlloc(own, &L.sq.lif, P));
    YC_TRY(devAlloc(own, &L.sq.att, P));
    YC_TRY(devAlloc(own, &L.qA, P));
    YC_TRY(devAlloc(own, &L.qH, P));
    YC_TRY(devAlloc(own, &L.qN, P));
    for (float4** r : {&L.ss.r0, &L.ss.r1, &L.ss.r2, &L.ss.r3, &L.ss.r4, &L.ss.r5, &L.ss.r6, &L.ss.r7}) YC_TRY(devAlloc(own, r, P));
    YC_TRY(devAlloc(own, &L.ctr, size_t(kCtrCount)));
    YC_TRY(rt::zero(ctx->st, L.ctr, kCtrCount * sizeof(uint32_t)));
    void* hp = nullptr;
    YC_TRY(rt::hostAlloc(&hp, kCtrCount * sizeof(uint32_t)));
    L.hCtr = static_cast<uint32_t*>(hp);
#ifndef YB_HOSTSIM
    uint2* sp = nullptr;
    YC_TRY(devAlloc(own, &sp, size_t(traceGridMax(ctx)) * kTraceBlock * kSpillEntries));
    L.spill = sp;
#endif
  }
  ctx->dCtr = ctx->lanes[0].ctr;
  ctx->dSpill = ctx->lanes[0].spill;
  YC_TRY(devAlloc(own, &ctx->dCounters, size_t(1)));
  YC_TRY(rt::zero(ctx->st, ctx->dCounters, sizeof(Counters)));
  YC_TRY(rt::sync(ctx->st));
  return YC_OK;
}

#ifndef YB_HOSTSIM
// The tail kernel's copies of the surviving paths' state (index-compatible with the lane's own arrays) and its private
// queues: allocated when a chunk first leaves paths to a tail (renders of depth 1 never do).
static int ensureTailStorage(yc_ctx* ctx, Lane& L) {
  if (L.tq) return YC_OK;
  auto& own = ctx->waveAllocs;
  const size_t P = L.capacity;
  YC_TRY(devAlloc(own, &L.ts.rayO, P));
  YC_TRY(devAlloc(own, &L.ts.rayD, P));
  YC_TRY(devAlloc(own, &L.ts.L, P));
  YC_TRY(devAlloc(own, &L.ts.att, P));
  YC_TRY(devAlloc(own, &L.ts.dim, P));
  YC_TRY(devAlloc(own, &L.ts.flags, P));
  YC_TRY(devAlloc(own, &L.ts.hitA, P));
  YC_TRY(devAlloc(own, &L.ts.hitB, P));
  YC_TRY(devAlloc(own, &L.tsq.o, size_t(kTailCapacity)));
  YC_TRY(devAlloc(own, &L.tsq.d, size_t(kTailCapacity)));
  YC_TRY(devAlloc(own, &L.tsq.lif, size_t(kTailCapacity)));
  YC_TRY(devAlloc(own, &L.tsq.att, size_t(kTailCapacity)));
  YC_TRY(devAlloc(own, &L.tq, size_t(kTailCapacity)));
  return YC_OK;
}
#endif

// ---------------------------------------------------------------------------------------
// frame + waves
// ---------------------------------------------------------------------------------------
// log2Int(float), math_base.hpp:156-160: the exponent, plus one when the significand is at least sqrt(2)'s
// (pbrt's rounding Log2Int) — e.g. 3 → 2, 5 → 2, 12 → 4, 100 → 7; exact for powers of two.
static uint32_t log2IntU(uint32_t value) {
  const float v = float(value);
  if (v < 1.0f) return 0;
  uint32_t bits;
  memcpy(&bits, &v, 4);
  const int32_t exponent = int32_t(bits >> 23) - 127;
  const uint32_t significand = bits & ((1u << 23) - 1u);
  return uint32_t(exponent + (significand >= 0x3504f3u ? 1 : 0));
}
static uint32_t roundUpPow2(uint32_t v) {  // math_base.hpp:164-170
  uint32_t p = 1;
  while (p < v) p <<= 1;
  return p;
}

extern "C" int yc_begin_frame(yc_ctx* ctx, const YcFrameDesc* f) {
  if (!ctx || !f) return YC_ERR_INVALID;
  YC_ENTER(ctx);
  if (!ctx->hasScene) return fail(ctx, YC_ERR_NO_SCENE, "yc_begin_frame before yc_upload_scene");
  if (!ctx->hasCamera) return fail(ctx, YC_ERR_STATE, "yc_begin_frame before yc_set_camera");
  if (f->width == 0 || f->height == 0 || f->width > 65535 || f->height > 65535 || f->tileSize == 0 ||
      f->totalSamples == 0 || f->estimator > YC_ESTIMATOR_GMONB || f->tonemap > YC_TONEMAP_AGX_PUNCHY)
    return fail(ctx, YC_ERR_INVALID, "bad frame description");
  const uint32_t shardCount = f->shardCount ? f->shardCount : 1;
  if (f->shardIndex >= shardCount) return fail(ctx, YC_ERR_INVALID, "shardIndex >= shardCount");
  YC_TRY(rt::sync(ctx->st));
  int rc = ensureWaveStorage(ctx);
  if (rc != YC_OK) return rc;
  // same geometry as the previous frame: keep the allocations and the pixel list, just clear
  const bool sameLayout = ctx->dHdr && ctx->frame.width == f->width && ctx->frame.height == f->height &&
                          ctx->frame.tileSize == f->tileSize && ctx->frame.shardIndex == f->shardIndex &&
                          ctx->frame.shardCount == shardCount;
  ctx->inFrame = false;
  const size_t frameTexels = size_t(f->width) * f->height;
  if (!sameLayout) {
    // a failure part-way must not leave a half-allocated frame that the next call's sameLayout test accepts:
    // the descriptor is committed only after every allocation succeeded
    freeFrame(ctx);
    ctx->frame = YcFrameDesc{};
    // tile list as TileRenderer::renderImpl builds it (tile-renderer.hpp:127-144), sharded by index
    ctx->pixels.clear();
    const uint32_t ts = f->tileSize;
    const uint32_t tilesX = (f->width + ts - 1) / ts, tilesY = (f->height + ts - 1) / ts;
    for (uint32_t ty = 0; ty < tilesY; ty++)
      for (uint32_t tx = 0; tx < tilesX; tx++) {
        const uint32_t index = ty * tilesX + tx;
        if (index % shardCount != f->shardIndex) continue;
        const uint32_t x0 = tx * ts, y0 = ty * ts;
        const uint32_t tw = std::min(ts, f->width - x0), th = std::min(ts, f->height - y0);
        for (uint32_t y = 0; y < th; y++)
          for (uint32_t x = 0; x < tw; x++) ctx->pixels.push_back((x0 + x) | ((y0 + y) << 16));
      }
    const size_t nPixNew = ctx->pixels.size();
    ctx->bucketCapacity = std::max<size_t>(nPixNew, 1);
    const char* e = nullptr;
    void* p = nullptr;
    if (!e && !(e = rt::alloc(&p, std::max<size_t>(nPixNew, 1) * 4))) ctx->dPixels = static_cast<uint32_t*>(p);
    if (!e && !(e = rt::alloc(&p, std::max<size_t>(nPixNew, 1) * 4))) ctx->dPixelsScratch = static_cast<uint32_t*>(p);
    if (!e && !(e = rt::alloc(&p, frameTexels * sizeof(float4)))) ctx->dHdr = static_cast<float4*>(p);
    if (!e && !(e = rt::alloc(&p, frameTexels * sizeof(float4)))) ctx->dLdr = static_cast<float4*>(p);
    if (!e && !(e = rt::alloc(&p, ctx->bucketCapacity * kMaxBuckets * sizeof(float4)))) ctx->dBuckets = static_cast<float4*>(p);
    if (!e) e = rt::h2d(ctx->st, ctx->dPixels, ctx->pixels.data(), nPixNew * 4);
    if (e) {
      freeFrame(ctx);
      return fail(ctx, YC_ERR_CUDA, "yc_begin_frame: %s", e);
    }
    ctx->bucketsDirty = true;  // fresh planes: clear below
  }
  ctx->frame = *f;
  ctx->frame.shardCount = shardCount;
  // finalize leaves every bucket it reads zeroed, so the planes only need clearing when an accumulate was not
  // followed by its finalize (an error or abort mid-wave, a partial-rectangle finalize) or when they are new
  if (ctx->bucketsDirty) {
    YC_TRY(rt::zero(ctx->st, ctx->dBuckets, ctx->bucketCapacity * kMaxBuckets * sizeof(float4)));
    ctx->bucketsDirty = false;
  }
  YC_TRY(rt::zero(ctx->st, ctx->dHdr, frameTexels * sizeof(float4)));
  YC_TRY(rt::zero(ctx->st, ctx->dLdr, frameTexels * sizeof(float4)));
  YC_TRY(rt::zero(ctx->st, ctx->dCounters, sizeof(Counters)));
  YC_TRY(rt::sync(ctx->st));
  ctx->launches = 0;
  ctx->gpuMs = ctx->extendMs = ctx->shadeMs = ctx->commMs = 0;
  ctx->extendLaunches = ctx->shadeLaunches = ctx->hitsShaded = 0;
  ctx->raysExtend = 0;
  ctx->inFrame = true;
  return YC_OK;
}

// One bounce of one lane's chunk: extend → sort → shade-miss → shade → shadow, then (unless it is the last
// possible bounce) an asynchronous read-back of the counters that size the next bounce.
template <bool ALPHA>
static int issueBounce(yc_ctx* ctx, Lane& L) {
  const uint32_t n = L.n;
  YC_TRY(rt::zero(L.st, L.ctr, kCtrCount * sizeof(uint32_t)));
  if (ctx->countTraversal) runExtend<ALPHA, true>(ctx, L, n);
  else runExtend<ALPHA, false>(ctx, L, n);
  rt::launchFor(L.st, n, SortMissK{ctx->ds, L.w, L.ps, L.qA, L.qH, L.ctr, ctx->dCounters});
  std::pair<rt::Event, rt::Event>* sev = nullptr;
  if (ctx->timeShade) {
    if (ctx->shadeEventsUsed == ctx->shadeEvents.size()) {
      ctx->shadeEvents.emplace_back();
      rt::eventCreate(ctx->shadeEvents.back().first);
      rt::eventCreate(ctx->shadeEvents.back().second);
    }
    sev = &ctx->shadeEvents[ctx->shadeEventsUsed++];
    rt::eventRecord(L.st, sev->first);
  }
  rt::launchFor<YB_RESOLVE_MIN_BLOCKS>(L.st, n, ResolveK{ctx->ds, L.ps, L.ss, L.qH, L.ctr});
  rt::launchFor<YB_SAMPLE_MIN_BLOCKS>(L.st, n, SampleK<ALPHA>{ctx->ds, L.w, L.ps, L.ss, L.qH, L.qA, L.qN, L.ctr, ctx->dCounters});
  rt::launchFor<YB_NEE_MIN_BLOCKS>(L.st, n, ShadeNeeK{ctx->ds, L.w, L.ss, L.sq, L.qH, L.qN, L.ctr});
  if (sev) rt::eventRecord(L.st, sev->second);
  if (ctx->countTraversal) runShadow<ALPHA, true>(ctx, L, n);
  else runShadow<ALPHA, false>(ctx, L, n);
  ctx->launches += 6;
  ctx->raysExtend += n;  // every queue entry is one closest-hit ray
  if (L.bounce + 1 < ctx->opts.maxDepth) {
    YC_TRY(rt::d2hAsync(L.st, L.hCtr, L.ctr, kCtrCount * sizeof(uint32_t)));
    rt::eventRecord(L.st, L.evCtr);
    L.waiting = true;
  } else {
    L.waiting = false;  // the bounce loop ends here whatever the counts are: no host round trip
    L.done = true;
  }
  return YC_OK;
}

template <bool ALPHA>
static int renderChunks(yc_ctx* ctx, const uint32_t* dList, uint32_t nPixCall, uint32_t sampleOffset, uint32_t waveSamples,
                        uint32_t m, uint32_t bucketShard, uint32_t bucketShardCount) {
  const YcFrameDesc& f = ctx->frame;
  WaveParams w{};
  w.cam = ctx->cam;
  // SobolSampler ctor (sampler.hpp:74-82) as TileRenderer calls it: (totalSamples, {tileSize, tileSize})
  w.smp.log2spp = log2IntU(f.totalSamples);
  w.smp.nBase4Digits = log2IntU(roundUpPow2(f.tileSize)) + (w.smp.log2spp + 1) / 2;
  w.smp.scrambler = ctx->opts.scrambler;
  w.smp.kind = ctx->opts.sampler;
  w.smp.strata = uint32_t(std::ceil(std::sqrt(double(f.totalSamples))));  // StratifiedSampler ctor, sampler.hpp:49-51
  memcpy(w.bg, f.background, sizeof w.bg);
  w.maxDepth = ctx->opts.maxDepth;
  w.pixelList = dList;
  const float exposureScale = std::exp2(ctx->cam.exposure);  // integrator.cpp:23

  // chunk list: pixel blocks x sample groups, each at most one lane's capacity of paths
  // Bucket sharding (bucketShardCount = G > 1): the wave's work is cut into units (estimator bucket b, pixel class c)
  // — class c = the c-th of G equal contiguous ranges of the pixel list — and this context takes the units with
  // (b + c) % G == bucketShard.  Every GPU gets one unit per bucket (balanced for any m, and each GPU sees every
  // part of the image), each (bucket, pixel) slot is written by exactly one GPU, with that bucket's samples
  // b, b + m, b + 2m, ... in sample order — the reference's rounding sequence — and everything else stays zero:
  // the per-GPU bucket buffers add up exactly.
  struct Chunk {
    uint32_t pixBase, nPix, sDone, K, stride;  // samples sDone, sDone + stride, ... (K of them) of the wave
  };
  std::vector<Chunk> chunks;
  const uint32_t cap = ctx->lanes[0].capacity;
  if (bucketShardCount <= 1) {
    const uint32_t B = std::min<uint32_t>(nPixCall, cap);
    const uint32_t Kmax = std::max<uint32_t>(1u, cap / B);
    for (uint32_t pixBase = 0; pixBase < nPixCall; pixBase += B) {
      const uint32_t nPix = std::min(B, nPixCall - pixBase);
      for (uint32_t sDone = 0; sDone < waveSamples;) {
        const uint32_t K = std::min(Kmax, waveSamples - sDone);
        chunks.push_back({pixBase, nPix, sDone, K, 1u});
        sDone += K;
      }
    }
  } else {
    const uint32_t G = bucketShardCount;
    for (uint32_t b = 0; b < m && b < waveSamples; b++) {
      const uint32_t c = (bucketShard + G - b % G) % G;
      const uint32_t p0 = uint32_t(uint64_t(c) * nPixCall / G), p1 = uint32_t(uint64_t(c + 1) * nPixCall / G);
      if (p1 == p0) continue;
      const uint32_t nb = (waveSamples - b + m - 1) / m;  // samples of the wave that fall into bucket b
      const uint32_t B = std::min<uint32_t>(p1 - p0, cap);
      const uint32_t Kmax = std::max<uint32_t>(1u, cap / B);
      for (uint32_t pixBase = p0; pixBase < p1; pixBase += B) {
        const uint32_t nPix = std::min(B, p1 - pixBase);
        for (uint32_t j = 0; j < nb;) {
          const uint32_t K = std::min(Kmax, nb - j);
          chunks.push_back({pixBase, nPix, b + j * m, K, m});
          j += K;
        }
      }
    }
  }
  if (chunks.empty()) return YC_OK;

  // A wave that follows a settled context starts after what is queued on the main stream (ev0).  A wave chained behind
  // a pending one (yc_render_wave_async) starts its chunks at once — their buffers are guarded by the lanes' own events
  // — and only its accumulates wait: for the previous wave's finalize, which reads and zeroes the bucket planes.
  for (int l = 0; l < kLanes; l++) {
    Lane& L = ctx->lanes[l];
    if (!ctx->wavesPending) rt::streamWaitEvent(L.st, ctx->ev0);
    rt::streamWaitEvent(L.side, ctx->wavesPending ? ctx->evFinal : ctx->ev0);
    L.active = false;
    L.accPending[0] = L.accPending[1] = false;
  }
  // A chunk that has left its lane and waits for its turn to be accumulated (chunk order).
  struct Finished {
    bool valid = false;
    int lane = 0, buf = 0;
    uint32_t pixBase = 0, nPix = 0, K = 0, sDone = 0, stride = 1;
  };
  std::vector<Finished> finished(chunks.size());
  auto allStreams = [&](auto&& fn) {
    for (int l = 0; l < kLanes; l++) fn(ctx->lanes[l].st), fn(ctx->lanes[l].side);
  };
  auto abortRequested = [&] { return ctx->abortFlag && *ctx->abortFlag != 0; };
  auto abortNow = [&] {
    // stop issuing, let what is in flight drain (the lanes' buffers are reused by the next call)
    allStreams([](rt::Stream& st) { rt::sync(st); });
    return fail(ctx, YC_ERR_ABORTED, "aborted");
  };
  // The chunk on lane L is complete as far as the lane's stream is concerned (`tail`: up to a per-path tail that the
  // side stream runs on copies): hand it to the side stream and free the lane.
  auto retire = [&](Lane& L, int l, bool tail) {
#ifndef YB_HOSTSIM
    if (tail) {
      rt::streamWaitEvent(L.st, L.evTail);  // the previous tail of this lane has let go of `ts` / `tq`
      rt::launchFor(L.st, L.n, TailGatherK{L.ps, L.ts, L.qA, L.tq});
      ctx->launches++;
    }
#endif
    rt::eventRecord(L.st, L.evChunk);
    rt::streamWaitEvent(L.side, L.evChunk);
#ifndef YB_HOSTSIM
    if (tail) {
      const dim3 tg((L.n + kTailBlock - 1) / kTailBlock);
      if (!ALPHA && ctx->wide)
        tailKernel<false, WideWalk><<<tg, kTailBlock, 0, L.side.s>>>(ctx->ds, L.w, L.ts, L.tsq, L.tq, L.n, L.bounce, ctx->dCounters, L.ps.L);
      else
        tailKernel<ALPHA, Bvh2Walk><<<tg, kTailBlock, 0, L.side.s>>>(ctx->ds, L.w, L.ts, L.tsq, L.tq, L.n, L.bounce, ctx->dCounters, L.ps.L);
      rt::eventRecord(L.side, L.evTail);
      ctx->launches++;
    }
#endif
    Finished& f = finished[L.chunk];
    f.valid = true, f.lane = l, f.buf = L.lSel;
    f.pixBase = L.w.pixBase, f.nPix = L.w.nPix, f.K = L.K, f.sDone = L.sDone, f.stride = L.w.sStrideM1 + 1u;
    L.accPending[L.lSel] = true;
    L.lSel ^= 1;
    L.active = false, L.done = false, L.waiting = false;
  };

  size_t next = 0, nextAcc = 0;
  const int lanesUsed = ctx->oneLane ? 1 : kLanes;
  rt::Event* lastAcc = nullptr;
  while (nextAcc < chunks.size()) {
    if (abortRequested()) return abortNow();
    // start chunks on idle lanes whose next radiance buffer is free (its previous chunk's accumulate is at least launched)
    for (int l = 0; l < lanesUsed && next < chunks.size(); l++) {
      Lane& L = ctx->lanes[l];
      if (L.active || L.accPending[L.lSel]) continue;
      const Chunk& c = chunks[next];
      L.active = true, L.done = false, L.waiting = false;
      L.chunk = uint32_t(next++);
      L.w = w;
      L.w.pixBase = c.pixBase, L.w.nPix = c.nPix, L.w.s0 = sampleOffset + c.sDone;
      L.w.sStrideM1 = c.stride - 1u;
      L.K = c.K, L.sDone = c.sDone;
      L.n = c.K * c.nPix;
      L.bounce = 0;
      L.ps.L = L.Lbuf[L.lSel];
      rt::streamWaitEvent(L.st, L.evSide[L.lSel]);  // the accumulate that read this buffer last
      rt::launchFor(L.st, L.n, RaygenK{L.w, L.ps, L.qA});
      ctx->launches++;
      if (ctx->opts.integrator == YC_INTEGRATOR_NAIVE) {
        runNaive<ALPHA>(ctx, L);  // the whole path in one launch: nothing to wait for
        ctx->launches++;
        retire(L, l, false);
        continue;
      }
      const int rc = issueBounce<ALPHA>(ctx, L);
      if (rc != YC_OK) return rc;
      if (L.done) retire(L, l, false);
    }
    // accumulate retired chunks in chunk order: Integrator::render adds a pixel's samples in sample order
    // (integrator.cpp:19-24), and the buckets' rounding sequence depends on it
    bool progressed = false;
    while (nextAcc < chunks.size() && finished[nextAcc].valid) {
      const Finished& f = finished[nextAcc];
      Lane& L = ctx->lanes[f.lane];
      if (lastAcc) rt::streamWaitEvent(L.side, *lastAcc);
      PathState acc = L.ps;
      acc.L = L.Lbuf[f.buf];
      rt::launchFor(L.side, f.nPix,
                    AccumulateK{acc, ctx->dBuckets, ctx->bucketCapacity, f.pixBase, f.nPix, f.K, f.sDone, f.stride, m, ctx->frame.estimator,
                                exposureScale});
      rt::eventRecord(L.side, L.evSide[f.buf]);
      lastAcc = &L.evSide[f.buf];
      L.accPending[f.buf] = false;
      ctx->launches++;
      nextAcc++;
      progressed = true;
    }
    if (nextAcc >= chunks.size()) break;
    if (next < chunks.size()) {
      bool canStart = false;
      for (int l = 0; l < lanesUsed; l++) canStart |= !ctx->lanes[l].active && !ctx->lanes[l].accPending[ctx->lanes[l].lSel];
      if (canStart) continue;  // a lane (or its buffer) was freed: give it the next chunk before blocking
    }
    // service whichever waiting lane's counters arrive first: they size its next bounce
    Lane* W = nullptr;
    int waiting = 0;
    for (int l = 0; l < kLanes; l++) waiting += ctx->lanes[l].active && ctx->lanes[l].waiting;
    if (!waiting) {
      if (progressed) continue;
      return fail(ctx, YC_ERR_STATE, "wavefront scheduler stalled");
    }
    int wl = 0;
    for (int spin = 0; !W; spin++) {
      for (int l = 0; l < kLanes && !W; l++) {
        Lane& L = ctx->lanes[l];
        if (L.active && L.waiting && (waiting == 1 || rt::eventReady(L.evCtr))) W = &L, wl = l;
      }
    }
    Lane& L = *W;
    rt::eventSync(L.evCtr);
    if (abortRequested()) return abortNow();
    L.waiting = false;
    ctx->hitsShaded += L.hCtr[kCtrHitCount];  // of the bounces whose counters come back (all but a path's last possible one)
    L.n = L.hCtr[kCtrNextCount];
    L.bounce++;
    if (L.n == 0 || L.bounce >= ctx->opts.maxDepth) {
      retire(L, wl, false);
      continue;
    }
#ifndef YB_HOSTSIM
    if (L.n <= ctx->tailThreshold) {
      if (const int trc = ensureTailStorage(ctx, L)) return trc;
      retire(L, wl, true);
      continue;
    }
#endif
    const int rc = issueBounce<ALPHA>(ctx, L);
    if (rc != YC_OK) return rc;
    if (L.done) retire(L, wl, false);
  }
  // the main stream continues (finalize) after the last accumulate, which waited for all earlier ones
  if (lastAcc) rt::streamWaitEvent(ctx->st, *lastAcc);
  YC_TRY(rt::lastError());
  return YC_OK;
}

// Pixel list of a call: the whole shard, or its intersection with `px` (uploaded to the scratch list).
static int wavePixels(yc_ctx* ctx, YcRect px, const uint32_t** dList, uint32_t* nPixCall) {
  const YcFrameDesc& f = ctx->frame;
  if (uint64_t(px.x) + px.w > f.width || uint64_t(px.y) + px.h > f.height)
    return fail(ctx, YC_ERR_INVALID, "pixel rectangle outside the frame");
  *dList = ctx->dPixels;
  *nPixCall = uint32_t(ctx->pixels.size());
  if (!(px.x == 0 && px.y == 0 && px.w == f.width && px.h == f.height)) {
    std::vector<uint32_t> sub;
    for (uint32_t v : ctx->pixels) {
      const uint32_t x = v & 0xffffu, y = v >> 16;
      if (x >= px.x && x < px.x + px.w && y >= px.y && y < px.y + px.h) sub.push_back(v);
    }
    *nPixCall = uint32_t(sub.size());
    YC_TRY(rt::h2d(ctx->st, ctx->dPixelsScratch, sub.data(), sub.size() * 4));
    *dList = ctx->dPixelsScratch;
  }
  return YC_OK;
}

static uint32_t waveBuckets(const YcFrameDesc& f, uint32_t waveSamples) {
  return f.estimator == YC_ESTIMATOR_MEAN ? 1u : uint32_t(estimatorBuckets(int(waveSamples), kMaxBuckets));
}

static int endTimedRegion(yc_ctx* ctx) {
  rt::eventRecord(ctx->st, ctx->ev1);
  return settleWaves(ctx);
}

// Waits for everything the context has issued (the main stream's last operation — a finalize, or the wait for the
// last accumulate — is ordered after all of a wave's work) and books the device time from the first unsettled wave's
// start to here.
static int settleWaves(yc_ctx* ctx) {
  ctx->wavesPending = false;
  YC_TRY(rt::sync(ctx->st));
  for (int l = 0; l < kLanes; l++) {  // idle already unless a wave was cut short (error, abort)
    YC_TRY(rt::sync(ctx->lanes[l].st));
    YC_TRY(rt::sync(ctx->lanes[l].side));
  }
  YC_TRY(rt::lastError());
  ctx->gpuMs += rt::eventElapsedMs(ctx->ev0, ctx->ev1);
  for (size_t i = 0; i < ctx->extendEventsUsed; i++) {
    ctx->extendMs += rt::eventElapsedMs(ctx->extendEvents[i].first, ctx->extendEvents[i].second);
    ctx->extendLaunches++;
  }
  ctx->extendEventsUsed = 0;
  for (size_t i = 0; i < ctx->shadeEventsUsed; i++) {
    ctx->shadeMs += rt::eventElapsedMs(ctx->shadeEvents[i].first, ctx->shadeEvents[i].second);
    ctx->shadeLaunches++;
  }
  ctx->shadeEventsUsed = 0;
  return YC_OK;
}

// The sample loop of a wave (Integrator::render, integrator.cpp:5-28) into the estimator buckets.
static int accumulateWave(yc_ctx* ctx, const uint32_t* dList, uint32_t nPixCall, uint32_t sampleOffset, uint32_t waveSamples,
                          uint32_t bucketShard, uint32_t bucketShardCount) {
  const uint32_t m = waveBuckets(ctx->frame, waveSamples);
  ctx->bucketsDirty = true;
  return ctx->ds.hasAlpha ? renderChunks<true>(ctx, dList, nPixCall, sampleOffset, waveSamples, m, bucketShard, bucketShardCount)
                          : renderChunks<false>(ctx, dList, nPixCall, sampleOffset, waveSamples, m, bucketShard, bucketShardCount);
}

// Estimator value of the wave + finishTile's blend and tonemap (tile-renderer.hpp:220-239).
static void finalizeWave(yc_ctx* ctx, const uint32_t* dList, uint32_t nPixCall, uint32_t waveSamples, uint32_t takenBefore) {
  const YcFrameDesc& f = ctx->frame;
  const uint32_t takenAfter = takenBefore + waveSamples;
  const float wCurrent = float(takenBefore) / float(takenAfter), wWave = float(waveSamples) / float(takenAfter);
  float4 *hdrRoot = nullptr, *ldrRoot = nullptr;
  if (ctx->comm && ctx->comm->direct) {
    Comm& c = *ctx->comm;
    // the copy the next yc_comm_reduce_frames publishes (noteWave has marked it stale if this wave is a partial one)
    if (dList == ctx->dPixels && !c.stale && c.frameTexels == size_t(f.width) * f.height) hdrRoot = c.hdrAll[c.epoch & 1u], ldrRoot = c.ldrAll[c.epoch & 1u];
  }
  rt::launchFor(ctx->st, nPixCall,
                FinalizeK{dList, ctx->dBuckets, ctx->bucketCapacity, ctx->dHdr, ctx->dLdr, hdrRoot, ldrRoot, f.width,
                          waveBuckets(f, waveSamples), f.estimator, waveSamples, f.tonemap, wCurrent, wWave});
  rt::eventRecord(ctx->st, ctx->evFinal);
  ctx->launches++;
  if (dList == ctx->dPixels) ctx->bucketsDirty = false;  // every plane this shard touches was read and zeroed
}

// Bookkeeping for the direct frame delivery of comm.cuh, from the ARGUMENTS of a finalizing call only — every
// participant makes the same calls, whether or not its shard has pixels in the rectangle, so all of them take the same
// decisions in the next yc_comm_reduce_frames (a collective must be entered by all or none).
static void noteWave(yc_ctx* ctx, YcRect px) {
  if (!ctx->comm) return;
  Comm& c = *ctx->comm;
  c.barrierSinceFinalize = false;
  const YcFrameDesc& f = ctx->frame;
  if (!(px.x == 0 && px.y == 0 && px.w == f.width && px.h == f.height) || c.frameTexels != size_t(f.width) * f.height) c.stale = true;
}

// One wave: the sample loop into the buckets, then estimator + blend + tonemap.  Chains behind waves that are still in
// flight (ctx->wavesPending) and leaves this one in flight.
static int issueWave(yc_ctx* ctx, YcRect px, uint32_t sampleOffset, uint32_t waveSamples, uint32_t takenBefore) {
  if (!ctx->inFrame) return fail(ctx, YC_ERR_STATE, "yc_render_wave before yc_begin_frame");
  noteWave(ctx, px);
  if (waveSamples == 0 || px.w == 0 || px.h == 0) return YC_OK;
  const uint32_t* dList;
  uint32_t nPixCall;
  if (const int prc = wavePixels(ctx, px, &dList, &nPixCall)) return prc;
  if (nPixCall == 0) return YC_OK;
  if (!ctx->wavesPending) rt::eventRecord(ctx->st, ctx->ev0);
  const int rc = accumulateWave(ctx, dList, nPixCall, sampleOffset, waveSamples, 0, 1);
  if (rc != YC_OK) {
    ctx->wavesPending = true;  // whatever was issued is waited for by the next entry point
    return rc;
  }
  finalizeWave(ctx, dList, nPixCall, waveSamples, takenBefore);
  rt::eventRecord(ctx->st, ctx->ev1);
  ctx->wavesPending = true;
  return YC_OK;
}

extern "C" int yc_render_wave(yc_ctx* ctx, YcRect px, uint32_t sampleOffset, uint32_t waveSamples, uint32_t takenBefore) {
  if (!ctx) return YC_ERR_INVALID;
  YC_ENTER(ctx);
  const int rc = issueWave(ctx, px, sampleOffset, waveSamples, takenBefore);
  const int src = ctx->wavesPending ? settleWaves(ctx) : YC_OK;
  return rc != YC_OK ? rc : src;
}

extern "C" int yc_render_wave_async(yc_ctx* ctx, YcRect px, uint32_t sampleOffset, uint32_t waveSamples, uint32_t takenBefore) {
  if (!ctx) return YC_ERR_INVALID;
  rt::useDevice(ctx->device);
  return issueWave(ctx, px, sampleOffset, waveSamples, takenBefore);
}

extern "C" int yc_wave_sync(yc_ctx* ctx) {
  if (!ctx) return YC_ERR_INVALID;
  YC_ENTER(ctx);
  return YC_OK;
}

extern "C" int yc_accumulate_wave(yc_ctx* ctx, YcRect px, uint32_t sampleOffset, uint32_t waveSamples, uint32_t bucketShard,
                                  uint32_t bucketShardCount) {
  if (!ctx) return YC_ERR_INVALID;
  YC_ENTER(ctx);
  if (!ctx->inFrame) return fail(ctx, YC_ERR_STATE, "yc_accumulate_wave before yc_begin_frame");
  if (bucketShardCount == 0 || bucketShard >= bucketShardCount) return fail(ctx, YC_ERR_INVALID, "bucket shard out of range");
  if (waveSamples == 0 || px.w == 0 || px.h == 0) return YC_OK;
  const uint32_t* dList;
  uint32_t nPixCall;
  if (const int prc = wavePixels(ctx, px, &dList, &nPixCall)) return prc;
  if (nPixCall == 0) return YC_OK;
  rt::eventRecord(ctx->st, ctx->ev0);
  const int rc = accumulateWave(ctx, dList, nPixCall, sampleOffset, waveSamples, bucketShard, bucketShardCount);
  if (rc != YC_OK) return rc;
  return endTimedRegion(ctx);
}

extern "C" int yc_finalize_wave(yc_ctx* ctx, YcRect px, uint32_t waveSamples, uint32_t takenBefore) {
  if (!ctx) return YC_ERR_INVALID;
  YC_ENTER(ctx);
  if (!ctx->inFrame) return fail(ctx, YC_ERR_STATE, "yc_finalize_wave before yc_begin_frame");
  noteWave(ctx, px);
  if (waveSamples == 0 || px.w == 0 || px.h == 0) return YC_OK;
  const uint32_t* dList;
  uint32_t nPixCall;
  if (const int prc = wavePixels(ctx, px, &dList, &nPixCall)) return prc;
  if (nPixCall == 0) return YC_OK;
  rt::eventRecord(ctx->st, ctx->ev0);
  finalizeWave(ctx, dList, nPixCall, waveSamples, takenBefore);
  return endTimedRegion(ctx);
}

extern "C" int yc_wave_buckets(yc_ctx* ctx, uint32_t waveSamples, uint32_t* m) {
  if (!ctx || !m) return YC_ERR_INVALID;
  YC_ENTER(ctx);
  if (!ctx->inFrame) return fail(ctx, YC_ERR_STATE, "no frame");
  *m = waveBuckets(ctx->frame, waveSamples);
  return YC_OK;
}

extern "C" int yc_bucket_device_ptrs(yc_ctx* ctx, void** buckets, size_t* bytes, uint32_t* planes, size_t* planePixels) {
  if (!ctx) return YC_ERR_INVALID;
  YC_ENTER(ctx);
  if (!ctx->inFrame) return fail(ctx, YC_ERR_STATE, "no frame");
  if (buckets) *buckets = ctx->dBuckets;
  if (bytes) *bytes = ctx->bucketCapacity * kMaxBuckets * sizeof(float4);
  if (planes) *planes = kMaxBuckets;
  if (planePixels) *planePixels = ctx->bucketCapacity;
  return YC_OK;
}

static int readStats(yc_ctx* ctx, YcStats* stats) {
  if (!stats) return YC_OK;
  Counters c{};
  if (ctx->dCounters) YC_TRY(rt::d2h(ctx->st, &c, ctx->dCounters, sizeof c));
  memset(stats, 0, sizeof *stats);
  stats->raysReference = c.raysReference;
  stats->raysExtend = ctx->raysExtend + c.raysExtend;
  stats->raysShadow = c.raysShadow;
  stats->boxTests = c.boxTests;
  stats->triTests = c.triTests;
  stats->kernelLaunches = ctx->launches;
  stats->gpuMs = ctx->gpuMs;
  stats->extendMs = ctx->extendMs;
  stats->shadeMs = ctx->shadeMs, stats->shadeLaunches = ctx->shadeLaunches, stats->hitsShaded = ctx->hitsShaded;
  stats->commMs = ctx->commMs;
  stats->extendLaunches = ctx->extendLaunches;
  return YC_OK;
}

extern "C" int yc_resolve(yc_ctx* ctx, float* hdrRGBA, float* ldrRGBA, YcStats* stats) {
  if (!ctx) return YC_ERR_INVALID;
  YC_ENTER(ctx);
  if (!ctx->inFrame) return fail(ctx, YC_ERR_STATE, "yc_resolve before yc_begin_frame");
  const size_t bytes = size_t(ctx->frame.width) * ctx->frame.height * sizeof(float4);
  if (hdrRGBA) YC_TRY(rt::d2h(ctx->st, hdrRGBA, ctx->dHdr, bytes));
  if (ldrRGBA) YC_TRY(rt::d2h(ctx->st, ldrRGBA, ctx->dLdr, bytes));
  return readStats(ctx, stats);
}

extern "C" int yc_frame_device_ptrs(yc_ctx* ctx, void** hdr, void** ldr, size_t* bytes) {
  if (!ctx) return YC_ERR_INVALID;
  YC_ENTER(ctx);
  if (!ctx->inFrame) return fail(ctx, YC_ERR_STATE, "no frame");
  if (hdr) *hdr = ctx->dHdr;
  if (ldr) *ldr = ctx->dLdr;
  if (bytes) *bytes = size_t(ctx->frame.width) * ctx->frame.height * sizeof(float4);
  return YC_OK;
}

extern "C" int yc_retonemap(yc_ctx* ctx) {
  if (!ctx) return YC_ERR_INVALID;
  YC_ENTER(ctx);
  if (!ctx->inFrame) return fail(ctx, YC_ERR_STATE, "no frame");
  rt::launchFor(ctx->st, ctx->frame.width * ctx->frame.height, RetonemapK{ctx->dHdr, ctx->dLdr, ctx->frame.tonemap});
  ctx->launches++;
  YC_TRY(rt::sync(ctx->st));
  YC_TRY(rt::lastError());
  return YC_OK;
}

extern "C" int yc_set_profiling(yc_ctx* ctx, int timeExtendKernel) {
  if (!ctx) return YC_ERR_INVALID;
  YC_ENTER(ctx);
  ctx->timeExtend = (timeExtendKernel & 1) != 0;
  ctx->countTraversal = (timeExtendKernel & 2) != 0;  // counting builds of extend / shadow (box / triangle tests)
  ctx->timeShade = (timeExtendKernel & 4) != 0;
  ctx->oneLane = (timeExtendKernel & 8) != 0;
  return YC_OK;
}

// ---------------------------------------------------------------------------------------
// ray-level hooks (parity tests + traversal microbench)
// ---------------------------------------------------------------------------------------
// The oracle's trace harness (oracle/ref_driver.cpp cmdTrace) restarts its sampler at pixel (0,0),
// sample 0 of a (16 spp, 64x64) SobolSampler before every ray; alpha-test draws use the same stream.
YB_DEV Sampler traceHookSampler() {
  SamplerConfig c;
  c.log2spp = 4;
  c.nBase4Digits = 6 + 2;
  c.scrambler = kScrambleFastOwen;
  c.kind = kSamplerSobol;
  c.strata = 4;
  Sampler s;
  s.start(c, 0, 0, 0);
  return s;
}

template <class Walk, bool NEE, bool ALPHA, bool COUNT, bool EARLY_OUT>
YB_DEV void traceOne(const DScene& sc, const YcRay& ray, bool useTMax, YcHit& out, TravStack& stack, TraceCounters& cnt) {
  Sampler smp = traceHookSampler();
  TraceState st;
  st.hit.t = (NEE || useTMax) ? ray.tmax : INFINITY;
  st.hit.node = kHitMiss;
  st.hit.u = st.hit.v = 0.0f;
  st.hit.prim = 0xffffffffu;
  st.hit.backSide = 0;
  st.attenuation = V3(1.0f);
  const V3 o(ray.o), d(ray.d);
  const bool did = traceScene<Walk, NEE, ALPHA, COUNT, EARLY_OUT>(sc, o, d, st, stack, &smp, cnt);
  out.t = st.hit.t;
  out.didHit = did ? 1u : 0u;
  out.prim = did ? st.hit.prim : 0xffffffffu;
  out.material = -1, out.lightIdx = -1, out.backSide = 0;
  for (int k = 0; k < 3; k++) out.p[k] = out.n[k] = out.tg[k] = 0.0f;
  out.uv[0] = out.uv[1] = 0.0f;
  out.attenuation[0] = st.attenuation.x, out.attenuation[1] = st.attenuation.y, out.attenuation[2] = st.attenuation.z;
  if (did) {
    const SurfaceHit s = resolveHit(sc, st.hit, o, d);
    out.material = s.material, out.lightIdx = s.lightIdx, out.backSide = st.hit.backSide;
    out.p[0] = s.p.x, out.p[1] = s.p.y, out.p[2] = s.p.z;
    out.n[0] = s.n.x, out.n[1] = s.n.y, out.n[2] = s.n.z;
    out.tg[0] = s.tg.x, out.tg[1] = s.tg.y, out.tg[2] = s.tg.z;
    out.uv[0] = s.uv.x, out.uv[1] = s.uv.y;
  }
}

// compact record of the device-resident variant: 20 bytes per hit (t, u, v, prim, node|backSide)
struct CompactHit {
  float t, u, v;
  uint32_t prim;
  int32_t node;
};

#ifdef YB_HOSTSIM
// The wide walk stops at an any-hit ray's first occluder, like shadowWideKernel; the reference-order walk keeps the
// reference's walk (ray-integrator.cpp:121).
template <bool NEE, bool ALPHA, bool COUNT, bool WIDE>
static void runTrace(yc_ctx* ctx, const YcRay* rays, uint32_t n, bool useTMax, YcHit* hits, CompactHit* compact) {
  HostStack hs;
  TraceCounters cnt;
  for (uint32_t i = 0; i < n; i++) {
    YcHit h;
    traceOne<std::conditional_t<WIDE, WideWalk, Bvh2Walk>, NEE, ALPHA, COUNT, NEE && WIDE>(ctx->ds, rays[i], useTMax, h, hs.ts, cnt);
    if (hits) hits[i] = h;
  }
  (void)compact;
  ctx->dCounters->boxTests += cnt.box;
  ctx->dCounters->triTests += cnt.tri;
}
#else
template <bool NEE, bool ALPHA, bool COMPACT>
struct TraceIO {
  DScene sc;
  const YcRay* rays;
  YcHit* hits;
  CompactHit* compact;
  int useTMax;
  __device__ __forceinline__ bool load(uint32_t i, V3& o, V3& d, float& tMax, Sampler& smp) const {
    const float4 a = __ldg(reinterpret_cast<const float4*>(rays) + 2 * size_t(i));
    const float4 b = __ldg(reinterpret_cast<const float4*>(rays) + 2 * size_t(i) + 1);
    o = V3(a.x, a.y, a.z);
    d = V3(b.x, b.y, b.z);
    tMax = (NEE || useTMax) ? b.w : INFINITY;
    smp = traceHookSampler();
    return true;
  }
  __device__ __forceinline__ void store(uint32_t i, const TraceState& st, bool did, const Sampler&) const {
    if (COMPACT) {
      CompactHit c;
      c.t = st.hit.t, c.u = st.hit.u, c.v = st.hit.v, c.prim = st.hit.prim;
      c.node = st.hit.node < 0 ? kHitMiss : int32_t(uint32_t(st.hit.node) | (st.hit.backSide ? kBackSideBit : 0u));
      compact[i] = c;
      return;
    }
    YcHit out;
    out.t = st.hit.t;
    out.didHit = did ? 1u : 0u;
    out.prim = did ? st.hit.prim : 0xffffffffu;
    out.material = -1, out.lightIdx = -1, out.backSide = 0;
    for (int k = 0; k < 3; k++) out.p[k] = out.n[k] = out.tg[k] = 0.0f;
    out.uv[0] = out.uv[1] = 0.0f;
    out.attenuation[0] = st.attenuation.x, out.attenuation[1] = st.attenuation.y, out.attenuation[2] = st.attenuation.z;
    if (did) {
      const float4 a = __ldg(reinterpret_cast<const float4*>(rays) + 2 * size_t(i));
      const float4 b = __ldg(reinterpret_cast<const float4*>(rays) + 2 * size_t(i) + 1);
      const SurfaceHit s = resolveHit(sc, st.hit, V3(a.x, a.y, a.z), V3(b.x, b.y, b.z));
      out.material = s.material, out.lightIdx = s.lightIdx, out.backSide = st.hit.backSide;
      out.p[0] = s.p.x, out.p[1] = s.p.y, out.p[2] = s.p.z;
      out.n[0] = s.n.x, out.n[1] = s.n.y, out.n[2] = s.n.z;
      out.tg[0] = s.tg.x, out.tg[1] = s.tg.y, out.tg[2] = s.tg.z;
      out.uv[0] = s.uv.x, out.uv[1] = s.uv.y;
    }
    hits[i] = out;
  }
};

template <bool NEE, bool ALPHA, bool COUNT, bool COMPACT>
__global__ void __launch_bounds__(kTraceBlock, YB_TRACE_MIN_BLOCKS) traceKernel(DScene sc, const YcRay* rays, uint32_t n, int useTMax, YcHit* hits,
                                                           CompactHit* compact, uint32_t* head, Counters* counters,
                                                           uint2* spill, TraceTuning tune) {
  TraceIO<NEE, ALPHA, COMPACT> io{sc, rays, hits, compact, useTMax};
  TraceCounters cnt;
  tracePersistent<Bvh2Walk, NEE, ALPHA, COUNT, false>(sc, io, n, head, spill, tune, cnt);
  flushCounts<COUNT>(counters, cnt);
}

// EARLY_OUT = NEE: an any-hit ray stops at its first occluder, like shadowWideKernel
template <bool NEE, bool COUNT, bool COMPACT>
__global__ void __launch_bounds__(kTraceBlock, YB_WIDE_MIN_BLOCKS) traceWideKernel(DScene sc, const YcRay* rays, uint32_t n, int useTMax, YcHit* hits,
                                                             CompactHit* compact, uint32_t* head, Counters* counters,
                                                             uint2* spill, TraceTuning tune) {
  TraceIO<NEE, false, COMPACT> io{sc, rays, hits, compact, useTMax};
  TraceCounters cnt;
  tracePersistent<WideWalk, NEE, false, COUNT, NEE>(sc, io, n, head, spill, tune, cnt);
  flushCounts<COUNT>(counters, cnt);
}

template <bool NEE, bool ALPHA, bool COUNT, bool WIDE>
static void runTrace(yc_ctx* ctx, const YcRay* rays, uint32_t n, bool useTMax, YcHit* hits, CompactHit* compact) {
  const auto kernel = WIDE ? (compact ? traceWideKernel<NEE, COUNT, true> : traceWideKernel<NEE, COUNT, false>)
                           : (compact ? traceKernel<NEE, ALPHA, COUNT, true> : traceKernel<NEE, ALPHA, COUNT, false>);
  kernel<<<traceGrid(ctx, n), kTraceBlock, 0, ctx->st.s>>>(ctx->ds, rays, n, useTMax, hits, compact, ctx->dCtr, ctx->dCounters,
                                                          static_cast<uint2*>(ctx->dSpill), tuning(ctx));
}
#endif

// Which walk a ray hook uses: the context's (YcOptions::traversal) unless the mode forces one; counting traces
// default to the reference-order walk (their box / triangle counts define the roofline's algorithmic bytes).
static int traceUsesWide(yc_ctx* ctx, int mode, bool* wide) {
  const bool count = (mode & YC_TRACE_COUNT) != 0;
  *wide = (mode & YC_TRACE_WIDE) ? true : (mode & YC_TRACE_REFERENCE_ORDER) ? false : (ctx->wide && !count);
  if (*wide && !ctx->ds.wideNodes) return fail(ctx, YC_ERR_STATE, "no wide BVH for this scene (alpha-tested materials, or traversal = reference order)");
  return YC_OK;
}

static void dispatchTrace(yc_ctx* ctx, int mode, bool wide, const YcRay* rays, uint32_t n, YcHit* hits, CompactHit* compact) {
  const bool nee = (mode & 0xf) == YC_TRACE_ANY, count = (mode & YC_TRACE_COUNT) != 0, alpha = ctx->ds.hasAlpha != 0;
  const bool useTMax = (mode & YC_TRACE_USE_TMAX) != 0;
#define YB_TR(N, A, C) runTrace<N, A, C, false>(ctx, rays, n, useTMax, hits, compact)
#define YB_TW(N, C) runTrace<N, false, C, true>(ctx, rays, n, useTMax, hits, compact)
  if (wide) {
    if (nee) count ? YB_TW(true, true) : YB_TW(true, false);
    else count ? YB_TW(false, true) : YB_TW(false, false);
  } else if (nee) {
    if (alpha) count ? YB_TR(true, true, true) : YB_TR(true, true, false);
    else count ? YB_TR(true, false, true) : YB_TR(true, false, false);
  } else {
    if (alpha) count ? YB_TR(false, true, true) : YB_TR(false, true, false);
    else count ? YB_TR(false, false, true) : YB_TR(false, false, false);
  }
#undef YB_TR
#undef YB_TW
}

extern "C" int yc_trace_device(yc_ctx* ctx, const void* raysDev, size_t n, int mode, void* hitsDev, int repeat, float* ms) {
  if (!ctx || !raysDev || !hitsDev || n > 0xffffffffull) return YC_ERR_INVALID;
  YC_ENTER(ctx);
  if (!ctx->hasScene) return fail(ctx, YC_ERR_NO_SCENE, "yc_trace_device before yc_upload_scene");
  int rc = ensureWaveStorage(ctx);
  if (rc != YC_OK) return rc;
  if (repeat < 1) repeat = 1;
  bool wide;
  if ((rc = traceUsesWide(ctx, mode, &wide)) != YC_OK) return rc;
  float total = 0.0f;
  for (int r = 0; r < repeat; r++) {
    YC_TRY(rt::zero(ctx->st, ctx->dCtr, kCtrCount * sizeof(uint32_t)));
    rt::eventRecord(ctx->st, ctx->ev0);
    dispatchTrace(ctx, mode, wide, static_cast<const YcRay*>(raysDev), uint32_t(n), nullptr, static_cast<CompactHit*>(hitsDev));
    rt::eventRecord(ctx->st, ctx->ev1);
    ctx->launches++;
    YC_TRY(rt::sync(ctx->st));
    YC_TRY(rt::lastError());
    total += rt::eventElapsedMs(ctx->ev0, ctx->ev1);
  }
  if (ms) *ms = total / float(repeat);
  return YC_OK;
}

extern "C" int yc_trace(yc_ctx* ctx, const YcRay* rays, size_t n, int mode, YcHit* hits, YcStats* stats) {
  if (!ctx || (n && (!rays || !hits)) || n > 0xffffffffull) return YC_ERR_INVALID;
  YC_ENTER(ctx);
  if (!ctx->hasScene) return fail(ctx, YC_ERR_NO_SCENE, "yc_trace before yc_upload_scene");
  int rc = ensureWaveStorage(ctx);
  if (rc != YC_OK) return rc;
  bool wide;
  if ((rc = traceUsesWide(ctx, mode, &wide)) != YC_OK) return rc;
  if (mode & YC_TRACE_COUNT) YC_TRY(rt::zero(ctx->st, ctx->dCounters, sizeof(Counters)));
  if (n) {
    void *dr = nullptr, *dh = nullptr;
    YC_TRY(rt::alloc(&dr, n * sizeof(YcRay)));
    const char* e = rt::alloc(&dh, n * sizeof(YcHit));
    if (e) {
      rt::release(dr);
      return fail(ctx, YC_ERR_CUDA, "alloc hits: %s", e);
    }
    e = rt::h2d(ctx->st, dr, rays, n * sizeof(YcRay));
    if (!e) e = rt::zero(ctx->st, ctx->dCtr, kCtrCount * sizeof(uint32_t));
    if (!e) {
      dispatchTrace(ctx, mode, wide, static_cast<const YcRay*>(dr), uint32_t(n), static_cast<YcHit*>(dh), nullptr);
      ctx->launches++;
      e = rt::d2h(ctx->st, hits, dh, n * sizeof(YcHit));
    }
    if (!e) e = rt::lastError();
    rt::release(dr);
    rt::release(dh);
    if (e) return fail(ctx, YC_ERR_CUDA, "yc_trace: %s", e);
  }
  return readStats(ctx, stats);
}

extern "C" int yc_device_alloc(yc_ctx* ctx, size_t bytes, void** out) {
  if (!ctx || !out) return YC_ERR_INVALID;
  YC_ENTER(ctx);
  YC_TRY(rt::alloc(out, bytes));
  return YC_OK;
}
extern "C" int yc_device_free(yc_ctx* ctx, void* p) {
  if (!ctx) return YC_ERR_INVALID;
  YC_ENTER(ctx);
  rt::sync(ctx->st);
  rt::release(p);
  return YC_OK;
}
extern "C" int yc_host_alloc(yc_ctx* ctx, size_t bytes, void** out) {
  if (!ctx || !out) return YC_ERR_INVALID;
  YC_ENTER(ctx);
  YC_TRY(rt::hostAlloc(out, bytes));
  return YC_OK;
}
extern "C" int yc_host_free(yc_ctx* ctx, void* p) {
  if (!ctx) return YC_ERR_INVALID;
  YC_ENTER(ctx);
  rt::hostRelease(p);
  return YC_OK;
}
extern "C" int yc_memcpy_h2d(yc_ctx* ctx, void* dst, const void* src, size_t bytes) {
  if (!ctx || !dst || !src) return YC_ERR_INVALID;
  YC_ENTER(ctx);
  YC_TRY(rt::h2d(ctx->st, dst, src, bytes));
  return YC_OK;
}
extern "C" int yc_memcpy_d2h(yc_ctx* ctx, void* dst, const void* src, size_t bytes) {
  if (!ctx || !dst || !src) return YC_ERR_INVALID;
  YC_ENTER(ctx);
  YC_TRY(rt::d2h(ctx->st, dst, src, bytes));
  return YC_OK;
}

// RayIntegrator::sample's rays (ray-integrator.cpp:11-18) for the current frame, sample-major.
struct PrimaryRayK {
  WaveParams w;
  YcRay* rays;
  YB_DEV void operator()(uint32_t i) const {
    uint32_t px, py, s;
    pathPixelSample(w, i, px, py, s);
    Sampler smp;
    smp.start(w.smp, px, py, s);
    V3 o, d;
    primaryRay(w.cam, smp, px, py, o, d);
    YcRay r;
    r.o[0] = o.x, r.o[1] = o.y, r.o[2] = o.z, r.tmin = kTMin;
    r.d[0] = d.x, r.d[1] = d.y, r.d[2] = d.z, r.tmax = INFINITY;
    rays[i] = r;
  }
};

extern "C" int yc_generate_primary_rays(yc_ctx* ctx, uint32_t sampleOffset, uint32_t spp, void* raysDev) {
  if (!ctx || !raysDev) return YC_ERR_INVALID;
  YC_ENTER(ctx);
  if (!ctx->inFrame) return fail(ctx, YC_ERR_STATE, "yc_generate_primary_rays before yc_begin_frame");
  const YcFrameDesc& f = ctx->frame;
  WaveParams w{};
  w.cam = ctx->cam;
  w.smp.log2spp = log2IntU(f.totalSamples);
  w.smp.nBase4Digits = log2IntU(roundUpPow2(f.tileSize)) + (w.smp.log2spp + 1) / 2;
  w.smp.scrambler = ctx->opts.scrambler;
  w.smp.kind = ctx->opts.sampler;
  w.smp.strata = uint32_t(std::ceil(std::sqrt(double(f.totalSamples))));  // StratifiedSampler ctor, sampler.hpp:49-51
  w.pixelList = ctx->dPixels;
  w.pixBase = 0, w.nPix = uint32_t(ctx->pixels.size()), w.s0 = sampleOffset;
  const uint64_t n = uint64_t(w.nPix) * spp;
  if (n > 0xffffffffull) return fail(ctx, YC_ERR_INVALID, "too many rays");
  rt::launchFor(ctx->st, uint32_t(n), PrimaryRayK{w, static_cast<YcRay*>(raysDev)});
  ctx->launches++;
  YC_TRY(rt::sync(ctx->st));
  YC_TRY(rt::lastError());
  return YC_OK;
}

extern "C" int yc_set_abort_flag(yc_ctx* ctx, const volatile int32_t* flag) {
  if (!ctx) return YC_ERR_INVALID;
  ctx->abortFlag = flag;
  return YC_OK;
}

// ---------------------------------------------------------------------------------------
// collectives (comm.cuh)
// ---------------------------------------------------------------------------------------
static void destroyComm(yc_ctx* ctx) {
  if (!ctx->comm) return;
  Comm& c = *ctx->comm;
#ifndef YB_HOSTSIM
  if (c.nccl) nccl().CommDestroy(c.nccl);
#endif
  detachCombinedFrames(ctx);
  rt::release(c.scratch);
  ctx->comm.reset();
}

#ifndef YB_HOSTSIM
#define YC_NCCL(expr)                                                                    \
  do {                                                                                   \
    const ncclResult_t r_ = (expr);                                                      \
    if (r_ != ncclSuccess) return fail(ctx, YC_ERR_CUDA, "%s: %s", #expr, nccl().GetErrorString(r_)); \
  } while (0)
#endif

extern "C" int yc_comm_unique_id(void* id128) {
  if (!id128) return YC_ERR_INVALID;
#ifdef YB_HOSTSIM
  return YC_ERR_UNSUPPORTED;
#else
  if (!nccl().ok) {
    fprintf(stderr, "yart_b200: %s\n", nccl().error.c_str());
    return YC_ERR_UNSUPPORTED;
  }
  ncclUniqueId id;
  if (nccl().GetUniqueId(&id) != ncclSuccess) return YC_ERR_CUDA;
  memcpy(id128, &id, sizeof id);
  return YC_OK;
#endif
}

extern "C" int yc_comm_init_rank(yc_ctx* ctx, int rank, int world, const void* id128) {
  if (!ctx || !id128 || world < 1 || rank < 0 || rank >= world) return YC_ERR_INVALID;
  YC_ENTER(ctx);
#ifdef YB_HOSTSIM
  return fail(ctx, YC_ERR_UNSUPPORTED, "the CPU build has no NCCL: use yc_comm_init_custom or yc_comm_init_all");
#else
  if (!nccl().ok) return fail(ctx, YC_ERR_UNSUPPORTED, "%s", nccl().error.c_str());
  destroyComm(ctx);
  ctx->comm = std::make_unique<Comm>();
  ctx->comm->rank = rank, ctx->comm->world = world;
  ncclUniqueId id;
  memcpy(&id, id128, sizeof id);
  YC_NCCL(nccl().CommInitRank(&ctx->comm->nccl, world, id, rank));
  return YC_OK;
#endif
}

extern "C" int yc_comm_init_all(yc_ctx** ctxs, int n) {
  if (!ctxs || n < 1) return YC_ERR_INVALID;
  for (int i = 0; i < n; i++)
    if (!ctxs[i]) return YC_ERR_INVALID;
  if (n > 1) {
    bool shared = false;  // two contexts on one GPU: NCCL refuses duplicate devices
    for (int i = 0; i < n; i++)
      for (int j = i + 1; j < n; j++) shared |= ctxs[i]->device == ctxs[j]->device;
#ifdef YB_HOSTSIM
    shared = true;  // the CPU build has no devices at all
#endif
    if (shared) {
      if (n > kGroupMax) return fail(ctxs[0], YC_ERR_INVALID, "at most %d contexts in an in-process group", kGroupMax);
      // the group's sums read every participant's buffer from one device: distinct devices need peer access
      for (int i = 0; i < n; i++)
        for (int j = 0; j < n; j++) {
          rt::useDevice(ctxs[i]->device);
          if (const char* e = rt::enablePeer(ctxs[i]->device, ctxs[j]->device))
            return fail(ctxs[0], YC_ERR_UNSUPPORTED, "in-process group over devices %d and %d: %s", ctxs[i]->device, ctxs[j]->device, e);
        }
      auto group = std::make_shared<HostGroup>();
      group->n = n;
      for (int i = 0; i < n; i++) {
        destroyComm(ctxs[i]);
        ctxs[i]->comm = std::make_unique<Comm>();
        ctxs[i]->comm->rank = i, ctxs[i]->comm->world = n, ctxs[i]->comm->group = group;
      }
      return YC_OK;
    }
  }
#ifdef YB_HOSTSIM
  destroyComm(ctxs[0]);
  ctxs[0]->comm = std::make_unique<Comm>();
  return YC_OK;
#else
  yc_ctx* ctx = ctxs[0];
  if (!nccl().ok) return fail(ctx, YC_ERR_UNSUPPORTED, "%s", nccl().error.c_str());
  std::vector<int> devs;
  std::vector<ncclComm_t> comms(size_t(n), nullptr);
  for (int i = 0; i < n; i++) devs.push_back(ctxs[i]->device);
  YC_NCCL(nccl().CommInitAll(comms.data(), n, devs.data()));
  for (int i = 0; i < n; i++) {
    destroyComm(ctxs[i]);
    ctxs[i]->comm = std::make_unique<Comm>();
    ctxs[i]->comm->rank = i, ctxs[i]->comm->world = n, ctxs[i]->comm->nccl = comms[size_t(i)];
  }
  return YC_OK;
#endif
}

extern "C" int yc_comm_init_custom(yc_ctx* ctx, int rank, int world, yc_collective_fn fn, void* user) {
  if (!ctx || !fn || world < 1 || rank < 0 || rank >= world) return YC_ERR_INVALID;
  destroyComm(ctx);
  ctx->comm = std::make_unique<Comm>();
  ctx->comm->rank = rank, ctx->comm->world = world, ctx->comm->custom = fn, ctx->comm->customUser = user;
  return YC_OK;
}

extern "C" int yc_comm_destroy(yc_ctx* ctx) {
  if (!ctx) return YC_ERR_INVALID;
  YC_ENTER(ctx);
  rt::sync(ctx->st);
  destroyComm(ctx);
  return YC_OK;
}

// Sum of `count` elements over all participants, in place on this context's stream; into `root` only when root >= 0
// (the other participants' buffers are then unspecified).
static int commSum(yc_ctx* ctx, void* buf, size_t count, int dtype, int root) {
  Comm& c = *ctx->comm;
  if (c.world == 1) return YC_OK;
  if (c.custom) {
    YC_TRY(rt::sync(ctx->st));  // the caller's collective knows nothing of our stream
    if (c.custom(buf, count, dtype, root, c.customUser) != 0) return fail(ctx, YC_ERR_CUDA, "the custom collective failed");
    return YC_OK;
  }
  if (c.group) {
    YC_TRY(rt::sync(ctx->st));  // this participant's buffer is final before the group meets
    const char* e = c.group->sum(c.rank, buf, [&](const GroupPtrs& bufs, int n) -> const char* {
#ifdef YB_HOSTSIM
      if (dtype == kCommF32) hostSum<float>(bufs, n, count, root);
      else if (dtype == kCommI32) hostSum<uint32_t>(bufs, n, count, root);  // wrap-around add of bit patterns: x + 0 is exact
      else hostSum<uint64_t>(bufs, n, count, root);
      return nullptr;
#else
      // the last arrival adds on its own stream; the contexts share a device (or peer access), so every pointer is valid here
      const int grid = int(std::min<size_t>((count + 255) / 256, size_t(ctx->smCount) * 8));
      if (dtype == kCommF32) groupSumKernel<float><<<grid, 256, 0, ctx->st.s>>>(bufs, n, count, root);
      else if (dtype == kCommI32) groupSumKernel<uint32_t><<<grid, 256, 0, ctx->st.s>>>(bufs, n, count, root);
      else groupSumKernel<unsigned long long><<<grid, 256, 0, ctx->st.s>>>(bufs, n, count, root);
      if (const char* se = rt::sync(ctx->st)) return se;
      return rt::lastError();
#endif
    });
    if (e) return fail(ctx, YC_ERR_CUDA, "in-process group sum: %s", e);
    return YC_OK;
  }
#ifndef YB_HOSTSIM
  const ncclDataType_t t = dtype == kCommF32 ? ncclFloat32 : dtype == kCommI32 ? ncclInt32 : ncclUint64;
  if (root < 0) YC_NCCL(nccl().AllReduce(buf, buf, count, t, ncclSum, c.nccl, ctx->st.s));
  else YC_NCCL(nccl().Reduce(buf, buf, count, t, ncclSum, root, c.nccl, ctx->st.s));
  return YC_OK;
#else
  return fail(ctx, YC_ERR_STATE, "communicator without a transport");
#endif
}

// Sum of n (<= 64) host values over all participants, in place.
static int commSumHost(yc_ctx* ctx, uint64_t* values, uint32_t n) {
  Comm& c = *ctx->comm;
  if (!c.scratch) {
    void* p = nullptr;
    YC_TRY(rt::alloc(&p, 64 * sizeof(uint64_t)));
    c.scratch = static_cast<uint64_t*>(p);
  }
  YC_TRY(rt::h2d(ctx->st, c.scratch, values, n * sizeof(uint64_t)));
  const int rc = commSum(ctx, c.scratch, n, kCommU64, -1);
  if (rc != YC_OK) return rc;
  YC_TRY(rt::d2h(ctx->st, values, c.scratch, n * sizeof(uint64_t)));
  c.barrierSinceFinalize = true;
  return YC_OK;
}

// Letting go of the root's combined frames.  An importer says so in the block itself before it closes its mapping; the
// root frees the block once every importer has (freeing memory that another process still maps is undefined), waits
// two seconds for that at most — a peer may have died — and then rather leaks the block than frees it.
static void detachCombinedFrames(yc_ctx* ctx) {
  Comm& c = *ctx->comm;
  if (c.imported) {
    const uint32_t one = 1;
    if (c.detached && c.rank >= 0 && c.rank < kGroupMax) rt::h2d(ctx->st, c.detached + c.rank, &one, sizeof one);
    rt::ipcClose(c.imported);
    rt::lastError();
    c.imported = nullptr;
  }
  if (c.block) {
    bool free_ = true;
    if (c.importers && c.detached) {
      free_ = false;
      for (int spin = 0; spin < 2000 && !free_; spin++) {
        uint32_t flags[kGroupMax] = {};
        if (rt::d2h(ctx->st, flags, c.detached, sizeof flags)) break;
        uint32_t n = 0;
        for (uint32_t f : flags) n += f != 0;
        free_ = n >= c.importers;
        if (!free_) std::this_thread::sleep_for(std::chrono::milliseconds(1));
      }
      if (!free_) fprintf(stderr, "yart_b200: a participant still maps the combined frames; leaving them allocated\n");
    }
    if (free_) rt::release(c.block);
    c.block = nullptr;
  }
  c.detached = nullptr;
  c.importers = 0;
  for (int k = 0; k < 2; k++) c.hdrAll[k] = c.ldrAll[k] = nullptr;
}

// (Re)creates the root's combined frames for the current frame size and finds out — collectively — whether every
// participant can address them (Comm::direct).  The root hands out {process id, device, address, exported handle} as a
// sum in which everybody else contributes zeros.
static int mapCombinedFrames(yc_ctx* ctx, int root, size_t texels) {
  Comm& c = *ctx->comm;
  detachCombinedFrames(ctx);
  c.frameTexels = texels, c.root = root, c.direct = false, c.stale = true, c.epoch = 0, c.cur = 0;
  const bool isRoot = c.rank == root;
  const size_t blockBytes = 4 * texels * sizeof(float4) + kGroupMax * sizeof(uint32_t);
  if (isRoot) {
    void* p = nullptr;
    YC_TRY(rt::alloc(&p, blockBytes));
    c.block = static_cast<float4*>(p);
    YC_TRY(rt::zero(ctx->st, c.block, blockBytes));
    YC_TRY(rt::sync(ctx->st));
  }
  auto carve = [&](float4* base) {
    for (int k = 0; k < 2; k++) c.hdrAll[k] = base + size_t(2 * k) * texels, c.ldrAll[k] = base + size_t(2 * k + 1) * texels;
    c.detached = reinterpret_cast<uint32_t*>(base + 4 * texels);
  };
  if (isRoot) carve(c.block);
  if (c.world == 1 || c.custom) return YC_OK;  // the caller's collective: nothing is known about the other side's memory

  constexpr uint32_t kWords = 3 + uint32_t((rt::kIpcHandleBytes + 7) / 8);
  static_assert(kWords <= 64, "payload must fit the staging buffer");
  uint64_t msg[kWords] = {};
  if (isRoot) {
    msg[0] = uint64_t(getpid()), msg[1] = uint64_t(ctx->device), msg[2] = uint64_t(reinterpret_cast<uintptr_t>(c.block));
    if (rt::ipcExport(c.block, &msg[3])) memset(&msg[3], 0, rt::kIpcHandleBytes), rt::lastError();
  }
  if (const int rc = commSumHost(ctx, msg, kWords)) return rc;
  uint64_t failed = 0;
  if (!isRoot) {
    float4* base = nullptr;
    if (msg[0] == uint64_t(getpid())) {  // another context of this process: plain peer access
      if (rt::enablePeer(ctx->device, int(msg[1]))) failed = 1, rt::lastError();
      else base = reinterpret_cast<float4*>(uintptr_t(msg[2]));
    } else {
      void* p = nullptr;
      if (rt::ipcImport(&p, &msg[3])) failed = 1, rt::lastError();
      else c.imported = p, base = static_cast<float4*>(p);
    }
    if (base) carve(base);
  }
  // YART_B200_FRAMES_REDUCE=1 (set for every participant) forces the summing path: for A/B measurements
  if (const char* e = getenv("YART_B200_FRAMES_REDUCE"))
    if (*e && *e != '0') failed = 1;
  uint64_t votes[2] = {failed, uint64_t(c.imported != nullptr)};
  if (const int rc = commSumHost(ctx, votes, 2)) return rc;
  c.direct = votes[0] == 0;
  if (isRoot) c.importers = uint32_t(votes[1]);
  if (!c.direct && !isRoot) detachCombinedFrames(ctx);  // (the root keeps its block: the summing path's destination)
  return YC_OK;
}

static int reduceFrames(yc_ctx* ctx, int root, bool async) {
  if (!ctx) return YC_ERR_INVALID;
  rt::useDevice(ctx->device);
  if (!ctx->comm) return fail(ctx, YC_ERR_STATE, "yc_comm_reduce_frames without a communicator");
  if (!ctx->inFrame) return fail(ctx, YC_ERR_STATE, "no frame");
  Comm& c = *ctx->comm;
  if (root < 0 || root >= c.world) return fail(ctx, YC_ERR_INVALID, "bad root");
  const size_t texels = size_t(ctx->frame.width) * ctx->frame.height;
#ifndef YB_HOSTSIM
  if (async && ctx->wavesPending && c.direct && !c.stale && c.nccl && c.frameTexels == texels && c.root == root) {
    // Chained behind waves in flight: the barrier is enqueued on the main stream after the wave's finalize kernel and
    // nobody waits for it here.  (The stores of wave k + 2 into this copy are issued after barrier k + 1, which the
    // root enters only once it has read what it wanted of wave k.)
    if (!c.barrierSinceFinalize) {
      if (!c.scratch) return fail(ctx, YC_ERR_STATE, "no staging buffer");
      if (const int rc = commSum(ctx, c.scratch, 1, kCommU64, -1)) return rc;
    }
    rt::eventRecord(ctx->st, ctx->ev1);
    c.barrierSinceFinalize = false;
    c.cur = int(c.epoch & 1u);
    c.epoch++;
    return YC_OK;
  }
#endif
  (void)async;
  if (ctx->wavesPending)
    if (const int rc = settleWaves(ctx)) return rc;
  if (c.frameTexels != texels || c.root != root) {
    if (const int rc = mapCombinedFrames(ctx, root, texels)) return rc;
  }
  rt::eventRecord(ctx->st, ctx->ev0);
  if (c.direct) {
    // Every finished pixel is already in the root's copy `epoch & 1` (FinalizeK stored it there), unless this context
    // has to catch up.  What is left is the guarantee that everybody's stores have landed: one small collective on
    // the streams that ran the finalize kernels — or none, if the caller has run one since (yc_comm_sum_u64).
    const int k = int(c.epoch & 1u);
    bool barrier = !c.barrierSinceFinalize;
    if (c.stale) {
      rt::launchFor(ctx->st, uint32_t(ctx->pixels.size()),
                    PushFramesK{ctx->dPixels, ctx->dHdr, ctx->dLdr, c.hdrAll[k], c.ldrAll[k], ctx->frame.width});
      ctx->launches++;
      c.stale = false;
      barrier = true;
    }
    if (barrier) {
      // the smallest collective there is, on the stream, no host values involved (the staging word's content is irrelevant)
      if (!c.scratch) {
        void* p = nullptr;
        YC_TRY(rt::alloc(&p, 64 * sizeof(uint64_t)));
        c.scratch = static_cast<uint64_t*>(p);
        YC_TRY(rt::zero(ctx->st, c.scratch, 64 * sizeof(uint64_t)));
      }
      if (const int rc = commSum(ctx, c.scratch, 1, kCommU64, -1)) return rc;
    }
    c.barrierSinceFinalize = false;
    c.cur = k;
    c.epoch++;
  } else {
    // out of place: the context's own frames keep blending its tiles in later waves
    float4 *hdr = c.hdrAll[0], *ldr = c.ldrAll[0];
    if (c.rank != root) {
      // a non-root participant of a summing transport needs a send buffer of its own
      if (!c.block) {
        void* p = nullptr;
        YC_TRY(rt::alloc(&p, 2 * texels * sizeof(float4)));
        c.block = static_cast<float4*>(p);
      }
      hdr = c.block, ldr = c.block + texels;
    }
    YC_TRY(rt::d2d(ctx->st, hdr, ctx->dHdr, texels * sizeof(float4)));
    YC_TRY(rt::d2d(ctx->st, ldr, ctx->dLdr, texels * sizeof(float4)));
    int rc = commSum(ctx, hdr, texels * 4, kCommF32, root);
    if (rc == YC_OK) rc = commSum(ctx, ldr, texels * 4, kCommF32, root);
    if (rc != YC_OK) return rc;
    c.cur = 0;
  }
  rt::eventRecord(ctx->st, ctx->ev1);
  YC_TRY(rt::sync(ctx->st));
  YC_TRY(rt::lastError());
  ctx->commMs += rt::eventElapsedMs(ctx->ev0, ctx->ev1);
  return YC_OK;
}

extern "C" int yc_comm_reduce_frames(yc_ctx* ctx, int root) { return reduceFrames(ctx, root, false); }
extern "C" int yc_comm_reduce_frames_async(yc_ctx* ctx, int root) { return reduceFrames(ctx, root, true); }

extern "C" int yc_comm_frames_direct(yc_ctx* ctx, int* direct) {
  if (!ctx || !direct) return YC_ERR_INVALID;
  if (!ctx->comm) return fail(ctx, YC_ERR_STATE, "yc_comm_frames_direct without a communicator");
  *direct = ctx->comm->direct ? 1 : 0;
  return YC_OK;
}

extern "C" int yc_resolve_combined(yc_ctx* ctx, float* hdrRGBA, float* ldrRGBA) {
  if (!ctx) return YC_ERR_INVALID;
  YC_ENTER(ctx);
  if (!ctx->comm || ctx->comm->root != ctx->comm->rank || !ctx->comm->hdrAll[0])
    return fail(ctx, YC_ERR_STATE, "yc_resolve_combined: not the root of a completed yc_comm_reduce_frames");
  const Comm& c = *ctx->comm;
  const size_t bytes = c.frameTexels * sizeof(float4);
  if (hdrRGBA) YC_TRY(rt::d2h(ctx->st, hdrRGBA, c.hdrAll[c.cur], bytes));
  if (ldrRGBA) YC_TRY(rt::d2h(ctx->st, ldrRGBA, c.ldrAll[c.cur], bytes));
  return YC_OK;
}

extern "C" int yc_comm_allreduce_buckets(yc_ctx* ctx, uint32_t waveSamples) {
  if (!ctx) return YC_ERR_INVALID;
  YC_ENTER(ctx);
  if (!ctx->comm) return fail(ctx, YC_ERR_STATE, "yc_comm_allreduce_buckets without a communicator");
  if (!ctx->inFrame) return fail(ctx, YC_ERR_STATE, "no frame");
  const size_t words = size_t(waveBuckets(ctx->frame, waveSamples)) * ctx->bucketCapacity * 4;
  rt::eventRecord(ctx->st, ctx->ev0);
  const int rc = commSum(ctx, ctx->dBuckets, words, kCommI32, -1);
  if (rc != YC_OK) return rc;
  rt::eventRecord(ctx->st, ctx->ev1);
  YC_TRY(rt::sync(ctx->st));
  YC_TRY(rt::lastError());
  ctx->commMs += rt::eventElapsedMs(ctx->ev0, ctx->ev1);
  return YC_OK;
}

extern "C" int yc_comm_sum_u64(yc_ctx* ctx, uint64_t* values, uint32_t n) {
  if (!ctx || !values || n == 0 || n > 64) return YC_ERR_INVALID;
  YC_ENTER(ctx);
  if (!ctx->comm) return fail(ctx, YC_ERR_STATE, "yc_comm_sum_u64 without a communicator");
  return commSumHost(ctx, values, n);
}

// ---- the reference's SAH BVH built on the device (bvh_build.cuh) -----------------------------------------------------
static thread_local std::string gBuildError;
extern "C" const char* yc_build_last_error() { return gBuildError.c_str(); }
static_assert(sizeof(YcBuildNode) == sizeof(yb::bvhb::RefNode), "YcBuildNode mirrors bvhb::RefNode");

extern "C" int yc_build_bvh_sah(int device, const float* positions, size_t nVerts, const uint32_t* faces4, size_t nTris,
                                YcBuildNode* nodes, uint32_t* nNodes, uint32_t* indices, uint32_t* levels) {
  if (!positions || !faces4 || !nodes || !nNodes || !indices || nTris == 0 || nVerts == 0) return YC_ERR_INVALID;
  for (size_t i = 0; i < nTris; i++)
    for (int k = 0; k < 3; k++)
      if (faces4[4 * i + k] >= nVerts) {
        gBuildError = "vertex index out of range";
        return YC_ERR_INVALID;
      }
  rt::Stream st;
  const char* traceEnv = getenv("YART_B200_BUILD_TRACE");
  const auto tA = std::chrono::high_resolution_clock::now();
  if (const char* e = rt::initStream(device, st)) {
    gBuildError = e;
    return YC_ERR_NO_DEVICE;
  }
  const auto tB = std::chrono::high_resolution_clock::now();
  const char* e = bvhb::build(st, positions, nVerts, faces4, nTris, reinterpret_cast<bvhb::RefNode*>(nodes), nNodes, indices, levels);
  const auto tC = std::chrono::high_resolution_clock::now();
  rt::destroy(st);
  if (traceEnv && *traceEnv && *traceEnv != '0')
    fprintf(stderr, "yart_b200 bvh build: device + stream %.1f ms, build incl. allocation %.1f ms, stream release %.1f ms\n",
            std::chrono::duration<double, std::milli>(tB - tA).count(), std::chrono::duration<double, std::milli>(tC - tB).count(),
            std::chrono::duration<double, std::milli>(std::chrono::high_resolution_clock::now() - tC).count());
  if (e) {
    gBuildError = e;
    return YC_ERR_CUDA;
  }
  return YC_OK;
}

#include "kat.cuh"
