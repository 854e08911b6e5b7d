/* yart_cuda.h — C ABI of the B200 wavefront path tracer that replaces yart's src/cpu
 * tile renderer (render hot path only).  Plain pointers and sizes; no C++/torch types.
 *
 * The reference (teofum/yart) has no FFI: its path sits behind C++ virtuals/templates.
 * Each entry point below names the reference interface it stands in for.  A maintainer's
 * `yart::cuda::WavefrontRenderer : yart::Renderer` would bind exactly these (INTEGRATION.md).
 *
 * Two layers live in the same shared library (libyart_b200.so):
 *   yc_*  device layer: flattened POD scene in, CUDA wavefront kernels, frames out.
 *   ys_* / yr_*  host layer: C mirror of yart's Scene / Camera / Renderer API
 *         (builds the SAH BVH exactly as src/core/bvh.hpp does and flattens it).
 *
 * All functions return YC_OK (0) or a negative YC_ERR_*; none throws across the ABI.
 * The reference is `noexcept` everywhere and signals failure by nullptr / silent return
 * (src/gltf/gltf.cpp:339, src/cpu/integrator.cpp:6); here the code is explicit.
 */
#ifndef YART_CUDA_H
#define YART_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define YC_OK 0
#define YC_ERR_INVALID (-1)   /* bad argument / inconsistent scene description */
#define YC_ERR_CUDA (-2)      /* CUDA runtime error (see yc_last_error) */
#define YC_ERR_NO_SCENE (-3)  /* render/trace before yc_upload_scene (reference: `if (!scene) return;`) */
#define YC_ERR_NO_DEVICE (-4) /* no usable CUDA device: there is NO CPU fallback */
#define YC_ERR_STATE (-5)     /* call order violated (e.g. render_wave before begin_frame) */
#define YC_ERR_IO (-6)
#define YC_ERR_UNSUPPORTED (-7) /* a variant this build of the library folds away: every sampler / scrambler other than
                                   YC_SAMPLER_SOBOL + YC_SCRAMBLER_FAST_OWEN needs libyart_b200_samplers.so (the same
                                   sources built with -DYB_RNG_SAMPLERS, same ABI) */

#define YC_ERR_ABORTED (-8)     /* the abort flag (yc_set_abort_flag / yr_abort) was raised: the wave was not finished */

#define YC_MAX_NODE_DEPTH 16

/* ---------------------------------------------------------------------------------------
 * Flattened scene (device layer input).  Host owns every pointer; yc_upload_scene copies.
 * ------------------------------------------------------------------------------------- */

/* Scene-graph node in DFS pre-order.  Replaces yart::Node (src/core/scene.hpp:11-64) as it is
 * walked by RayIntegrator::testNode (src/cpu/ray-integrator.cpp:20-54). */
typedef struct YcNode {
  float inv[12];  /* rows 0..2 of Transform::m_inverseTransform (row-major 3x4) */
  float fwd[12];  /* rows 0..2 of Transform::m_transform */
  float nrm[9];   /* Transform::m_normalTransform = transpose(float3x3(inverse)) */
  float bmin[3], bmax[3]; /* Node::boundingBox(), node object space */
  int32_t mesh;   /* index into meshes, -1 = none */
  int32_t parent; /* -1 for the root (node 0) */
  int32_t skip;   /* index of the first node after this node's subtree */
  int32_t depth;  /* root = 0; must be < YC_MAX_NODE_DEPTH */
  int32_t identityChain; /* 1 iff this node's and all its ancestors' transforms are exactly the identity */
} YcNode;

/* One inner BVH node with BOTH children's bounds inlined (64 B = 4 x 128-bit loads).
 * Same tree, same child order and same boxes as yart::BVHNode (src/core/bvh.hpp:21-33):
 * child 0 is `left`, child 1 is `left + 1`.
 * ref: inner child → index of its YcBvhNode (relative to the mesh's first node);
 *      leaf child  → 0x80000000 | index of its first YcBvhTri (relative to the mesh's first tri);
 *      the leaf's triangles follow contiguously, the last one carries YC_TRI_LAST. */
typedef struct YcBvhNode {
  float c0min[3], c0max[3];
  float c1min[3], c1max[3];
  uint32_t ref0, ref1;
  uint32_t pad0, pad1;
} YcBvhNode;

#define YC_REF_LEAF 0x80000000u
#define YC_TRI_LAST 1u        /* last triangle of its leaf */
#define YC_TRI_ALPHA 2u       /* material has alpha texels < 255 (parametric.cpp:57-61) */
#define YC_TRI_TRANSPARENT 4u /* material.transparent() (parametric.cpp:80-82) */

/* Leaf-ordered triangle record (48 B = 3 x 128-bit loads): positions pre-gathered in
 * BVH::m_indices order so a leaf is one contiguous run. */
typedef struct YcBvhTri {
  float p0[3], p1[3], p2[3];
  uint32_t prim;  /* original triangle index in the mesh (what Hit::idx holds) */
  uint32_t flags; /* YC_TRI_* */
  uint32_t pad;
} YcBvhTri;

typedef struct YcMesh {
  float rootMin[3], rootMax[3]; /* BVH root bounds (tested first, ray-integrator.cpp:98) */
  uint32_t rootRef;             /* like YcBvhNode::ref (root may itself be a leaf) */
  uint32_t nodeOffset;          /* first YcBvhNode of this mesh in YcScene::bvhNodes */
  uint32_t triOffset;           /* first YcBvhTri of this mesh in YcScene::bvhTris */
  uint32_t vertOffset;          /* first vertex in the vertex arrays */
  uint32_t primOffset;          /* first primitive in primIndices / primMaterial / primLight */
  uint32_t nTris, nVerts, nInner;
} YcMesh;

/* ParametricBSDF parameters (src/bsdf/parametric.hpp:15-36 + derived members :48-76). */
typedef struct YcMaterial {
  float base[3];
  float metallic, roughness, transmission, ior;
  float anisotropic, clearcoat, clearcoatRoughness;
  float emission[3];
  float normalScale; /* stored, never applied — as in the reference (core/bsdf.cpp:46-56) */
  float volumeColor[3];
  float volumeDensity;
  float localRotation[9]; /* float3x3(float4x4::rotation(-anisoRotation, z)) */
  float invRotation[9];   /* float3x3(float4x4::rotation(+anisoRotation, z)) */
  int32_t baseTex, mrTex, transTex, normalTex, ccTex, emisTex; /* -1 = none */
  int32_t thinTransmission, hasAlpha, hasEmission;
  int32_t pad;
} YcMaterial;

/* Texture<T,C> (src/core/texture.hpp:21-52).  u8 textures index texelsU8, float ones texelsF32. */
typedef struct YcTexture {
  uint64_t offset; /* element offset into texelsU8 / texelsF32 */
  uint32_t width, height, channels;
  uint32_t isFloat;
  uint32_t type; /* 0 LinearRGB, 1 sRGB (gamma-2 storage), 2 NonColor */
  uint32_t pad;
} YcTexture;

#define YC_LIGHT_AREA 0
#define YC_LIGHT_IMAGE_INFINITE 1
#define YC_LIGHT_UNIFORM_INFINITE 2

/* Light (src/core/light.hpp).  Area lights carry their triangle (mesh space) so that
 * AreaLight::sample (light.cpp:46-72) needs no mesh lookup. */
typedef struct YcLight {
  int32_t type;
  int32_t twoSided;
  float emission[3]; /* area / uniform */
  float area;        /* AreaLight::m_area (transformed triangle) */
  float power;       /* Light::power() */
  float p0[3], p1[3], p2[3]; /* mesh-space vertices */
  float n0[3], n1[3], n2[3]; /* mesh-space vertex normals */
  float fwd[12], nrm[9];     /* Light::m_transform (area) */
  /* infinite lights */
  float sceneRadius, surfaceArea;
  float Lavg[3];
  float envFwd[12], envInv[12]; /* ImageInfiniteLight::transform (public member) */
  int32_t hdrTex;
  uint32_t distW, distH;        /* PiecewiseConstant2D resolution */
  uint64_t distOffset;          /* float offset into YcScene::envDist of this light's block:
                                   func[W*H] cdf[(W+1)*H] rowIntegral[H] mfunc[H] mcdf[H+1] mIntegral[1] */
} YcLight;

typedef struct YcScene {
  const YcNode* nodes;       uint32_t nNodes;
  const YcMesh* meshes;      uint32_t nMeshes;
  const YcBvhNode* bvhNodes; uint64_t nBvhNodes;
  const YcBvhTri* bvhTris;   uint64_t nBvhTris;
  /* vertex attributes (all meshes concatenated) */
  const float* positions;    /* 3 per vertex */
  const float* normals;      /* 3 per vertex */
  const float* tangents;     /* 4 per vertex */
  const float* uvs;          /* 2 per vertex */
  uint64_t nVerts;
  /* primitives in original order (all meshes concatenated) */
  const uint32_t* primIndices; /* 3 per primitive, mesh-local vertex indices */
  const uint32_t* primMaterial;
  const int32_t* primLight;    /* Mesh::lightIdx, -1 = none */
  uint64_t nPrims;
  const YcMaterial* materials; uint32_t nMaterials;
  const YcTexture* textures;   uint32_t nTextures;
  const uint8_t* texelsU8;     uint64_t nTexelsU8;
  const float* texelsF32;      uint64_t nTexelsF32;
  const YcLight* lights;       uint32_t nLights;
  const float* envDist;        uint64_t nEnvDist;
  /* PowerLightSampler (src/core/light-sampler.cpp:32-93) */
  const uint32_t* infiniteLights; uint32_t nInfinite; /* scene light indices */
  const uint32_t* areaLights;     uint32_t nArea;     /* scene light indices, m_lights order */
  const float* lightPowerCdf;                         /* m_lightPowers (running sums), nArea */
  float totalPower;
  /* data tables (values dumped from the reference build, see yart_b200/data/README) */
  const float* lutTables;   /* 14112 floats, order documented in csrc/luts.cuh */
  int32_t hasAlpha;         /* any material with hasAlpha */
} YcScene;

/* Derived camera members (src/core/camera.hpp:17-22, computed by calcDerivedProperties :25-59). */
typedef struct YcCamera {
  float position[3];
  float topLeftPixel[3];
  float pixelDeltaU[3], pixelDeltaV[3];
  float frameX[3], frameY[3], frameZ[3]; /* m_cameraFrame */
  float apertureRadius;
  uint32_t apertureSides;
  float exposure;
} YcCamera;

typedef struct YcOptions {
  uint32_t maxDepth;        /* RayIntegrator::m_maxDepth (default 30) */
  uint32_t maxPathsInFlight; /* wavefront capacity; 0 = default (8 Mi paths) */
  /* Warp-scheduling knobs of the traversal kernels (0 = default); they never change results:
   * traceRefillMin — idle lanes at which a warp fetches new rays (default 8);
   * traceInnerMin  — lanes on inner nodes below which a warp leaves the inner-node loop (default 20). */
  uint32_t traceRefillMin, traceInnerMin;
  /* Surviving paths of a chunk at which its remaining bounces go to the per-path tail kernel
   * (0 = default 16384, 0xffffffff = never).  Never changes results. */
  uint32_t tailThreshold;
  /* The `Integrator` template argument of TileRenderer (src/main.cpp:17): YC_INTEGRATOR_MIS =
   * cpu::MISIntegrator (the measured path), YC_INTEGRATOR_NAIVE = cpu::NaiveIntegrator
   * (src/cpu/naive-integrator.cpp: BSDF sampling only, maxDepth + 1 segments, at most 63). */
  uint32_t integrator;
  /* The scrambler R of the `Sampler = SobolSampler<R>` template argument (src/main.cpp:16):
   * FastOwenScrambler (the measured path), OwenScrambler or BinaryPermuteScrambler (src/core/scrambler.hpp:35-85). */
  uint32_t scrambler;
  /* Entries of the traversal kernels' shared-memory stack actually used (0 = default, all 25); the rest goes to
   * the global spill area.  Never changes results; tests shrink it to exercise the spill path. */
  uint32_t sharedStackEntries;
  /* The `Sampler` template argument of TileRenderer (src/main.cpp:16): YC_SAMPLER_SOBOL = SobolSampler<R> with the
   * scrambler above (the measured path), YC_SAMPLER_NAIVE = NaiveSampler, YC_SAMPLER_STRATIFIED = StratifiedSampler
   * (src/core/sampler.cpp:5-50; xoshiro256++ seeded per pixel sample, re-derived per draw from the dimension). */
  uint32_t sampler;
  /* YC_LIGHT_SAMPLER_* — the m_lightSampler member of MISIntegrator (mis-integrator.hpp:20 hard-codes
   * PowerLightSampler; UniformLightSampler, light-sampler.cpp:11-31, is its alternative; variants build only). */
  uint32_t lightSampler;
  /* YC_TRAVERSAL_* — how RayIntegrator::testBVH (ray-integrator.cpp:84-160) is walked:
   *   AUTO             the 4-wide collapsed BVH (csrc/wide_bvh.cuh) for scenes without alpha-tested materials,
   *                    the reference-order BVH2 walk otherwise;
   *   REFERENCE_ORDER  always the BVH2 walk: same boxes, same order, same two-rounding slab test as the reference —
   *                    every hit, frame and ray count is bit-identical to the reference;
   *   WIDE             the wide walk or YC_ERR_UNSUPPORTED at yc_upload_scene (alpha-tested materials: the order of
   *                    triangle tests would move sampler draws).
   * The wide walk tests the reference's triangles with the reference's arithmetic and differs only in box culling
   * (hit ids / t identical except last-bit ties and box-boundary hits; frames within the north-star tolerance). */
  uint32_t traversal;
  uint32_t reserved;
} YcOptions;

#define YC_INTEGRATOR_MIS 0
#define YC_INTEGRATOR_NAIVE 1
#define YC_SCRAMBLER_FAST_OWEN 0
#define YC_SCRAMBLER_OWEN 1
#define YC_SCRAMBLER_BINARY_PERMUTE 2
#define YC_LIGHT_SAMPLER_POWER 0
#define YC_LIGHT_SAMPLER_UNIFORM 1
#define YC_SAMPLER_SOBOL 0
#define YC_SAMPLER_NAIVE 1
#define YC_SAMPLER_STRATIFIED 2
#define YC_TRAVERSAL_AUTO 0
#define YC_TRAVERSAL_REFERENCE_ORDER 1
#define YC_TRAVERSAL_WIDE 2

typedef struct YcRect { uint32_t x, y, w, h; } YcRect;

#define YC_TONEMAP_NONE 0
#define YC_TONEMAP_AGX 1
#define YC_TONEMAP_AGX_GOLDEN 2
#define YC_TONEMAP_AGX_PUNCHY 3

#define YC_ESTIMATOR_GMON 0 /* what Integrator::render instantiates (integrator.cpp:17) */
#define YC_ESTIMATOR_MON 1
#define YC_ESTIMATOR_MEAN 2
#define YC_ESTIMATOR_GMONB 3 /* GMoNbEstimator, estimator.hpp:94-141: mean when the Gini index <= 0.25, else median of means */

typedef struct YcFrameDesc {
  uint32_t width, height;
  uint32_t totalSamples; /* TileRenderer::samples: fixes the sampler's log2spp */
  uint32_t tileSize;     /* TileRenderer::tileSize: fixes the sampler's nBase4Digits */
  float background[3];   /* Renderer::backgroundColor */
  uint32_t tonemap;      /* YC_TONEMAP_* */
  uint32_t estimator;    /* YC_ESTIMATOR_* */
  /* multi-GPU: this context renders only tiles whose row-major index % shardCount == shardIndex
   * (tile list as in tile-renderer.hpp:127-144); other pixels stay 0 so frames sum across GPUs. */
  uint32_t shardIndex, shardCount;
} YcFrameDesc;

typedef struct YcStats {
  uint64_t raysReference;   /* reference definition: path segments + unoccluded non-zero-f NEE rays
                               (mis-integrator.cpp:22,126) */
  uint64_t raysExtend;      /* closest-hit rays traced */
  uint64_t raysShadow;      /* any-hit rays traced */
  uint64_t samples;         /* pixel samples taken since begin_frame, counted while adaptive sampling is on (ΣS of
                               yc_resolve_adaptive); 0 otherwise */
  uint64_t kernelLaunches;  /* CUDA kernels launched by this context since begin_frame */
  double gpuMs;             /* CUDA-event time spent inside yc_render_wave since begin_frame */
  uint64_t boxTests, triTests; /* only filled by counting traces (yc_trace with YC_TRACE_COUNT): the reference-order
                                  walk's tests unless YC_TRACE_WIDE is OR-ed in (then: wide child boxes tested) */
  double extendMs;          /* CUDA-event time of the extend (closest-hit) launches, when yc_set_profiling(1) */
  uint64_t extendLaunches;
  double shadeMs;           /* CUDA-event time of the surface-shading launches, when yc_set_profiling(4) */
  uint64_t shadeLaunches;
  uint64_t hitsShaded;      /* queue entries those launches shaded */
  double commMs;            /* CUDA-event time of the yc_comm_* data collectives since begin_frame */
} YcStats;

/* Adaptive sampling parameters (yc_set_adaptive, yr_set_adaptive). */
typedef struct YcAdaptive {
  float threshold;     /* a pixel stops once every e of its neighbourhood is below it; finite, >= 0 (0: none ever stops) */
  uint32_t minSamples; /* samples a pixel takes at least */
  float lumaFloor;     /* the denominator's floor: finite, > 0 */
  uint32_t reserved;
} YcAdaptive;

typedef struct YcRay { float o[3], tmin, d[3], tmax; } YcRay;

/* What the reference's Hit holds after testNode (src/cpu/hit.hpp:8-17). */
typedef struct YcHit {
  float t;
  uint32_t prim;     /* Hit::idx; 0xffffffff on miss */
  int32_t material;  /* index of Hit::bsdf, -1 on miss */
  int32_t lightIdx;
  uint32_t backSide;
  uint32_t didHit;
  float p[3], n[3], tg[3], uv[2];
  float attenuation[3];
} YcHit;

#define YC_TRACE_CLOSEST 0
#define YC_TRACE_ANY 1     /* NEE ray: Ray::nee = true, hit.t preset to tmax */
#define YC_TRACE_COUNT 16  /* OR-ed in: also count box / triangle tests into YcStats */
#define YC_TRACE_USE_TMAX 32 /* OR-ed in (closest): preset hit.t = ray.tmax instead of infinity */
#define YC_TRACE_REFERENCE_ORDER 64 /* OR-ed in: force the reference-order BVH2 walk for this call */
#define YC_TRACE_WIDE 128           /* OR-ed in: force the 4-wide walk (YC_ERR_STATE if the scene has none) */

typedef struct yc_ctx yc_ctx;

/* --- device layer ------------------------------------------------------------------- */
/* Replaces constructing a cpu::TileRenderer (src/cpu/tile-renderer.hpp:34-38). */
int yc_create(int device, const YcOptions* opts, yc_ctx** out);
void yc_destroy(yc_ctx* ctx);
const char* yc_last_error(const yc_ctx* ctx);
/* Replaces `renderer.scene = scene` (src/core/renderer.hpp:53). */
int yc_upload_scene(yc_ctx* ctx, const YcScene* scene);
/* Replaces the `const Camera&` the renderer holds (src/core/renderer.hpp:97).  yc_set_cameras(ctx, cam, 1). */
int yc_set_camera(yc_ctx* ctx, const YcCamera* cam);
/* Several views of the scene in one frame: n cameras (1 <= n <= 65535; YC_ERR_INVALID otherwise or for NULL) that share
 * the YcFrameDesc — size, samples, tile size, tonemap, estimator, background.  Each view is the frame its camera renders
 * alone, bit for bit (HDR, LDR, AOVs; the ray counts of YcStats add up over the views): the sampler depends on the
 * view-local pixel, the sample index and the frame's totalSamples / tileSize only.
 *   Layout: the views are stacked by rows.  View v occupies rows [v·height, (v+1)·height) of a frame of width x
 *     (height·n) texels: every frame and AOV plane is [n][height][width][4] floats.  YcRect arguments are in these
 *     stacked rows (a rectangle may span views); yc_generate_primary_rays writes the rays of every view.
 *   Tiles: the tile list is the reference's (tile-renderer.hpp:127-144) of each view, view after view; tile k of that
 *     list goes to shard k % shardCount.
 *   The view count of a frame is fixed by yc_begin_frame from the cameras set then.  Setting the same number of cameras
 *     later is allowed (the next wave uses them); after a different number, yc_render_wave[_async], yc_accumulate_wave,
 *     yc_finalize_wave and yc_generate_primary_rays return YC_ERR_STATE until the next yc_begin_frame.
 *   A frame holds at most 2^32 texels (YC_ERR_INVALID from yc_begin_frame). */
int yc_set_cameras(yc_ctx* ctx, const YcCamera* cams, uint32_t n);
/* Replaces TileRenderer::renderImpl's state reset (tile-renderer.hpp:118-124). */
int yc_begin_frame(yc_ctx* ctx, const YcFrameDesc* frame);
/* Replaces one wave of the worker loop + finishTile for every tile
 * (tile-renderer.hpp:161-191, 205-239; Integrator::render, integrator.cpp:5-28):
 * takes samples [sampleOffset, sampleOffset + waveSamples) of every pixel in `pixels`,
 * runs the per-wave estimator, blends into the HDR frame with sample-count weights
 * (takenBefore = samples already blended) and tonemaps. */
int yc_render_wave(yc_ctx* ctx, YcRect pixels, uint32_t sampleOffset, uint32_t waveSamples,
                   uint32_t takenBefore);
/* The same wave, left in flight: the call returns once the wave's last chunk has been handed to the GPU, and the next
 * yc_render_wave_async starts its chunks while this wave's per-path tails, bucket sums and finalize kernel still run
 * (the results are the same bits: accumulation stays in sample order and a wave's finalize precedes the next wave's
 * first bucket sum).  yc_wave_sync — or any other entry point — waits for the waves in flight; the frames, statistics
 * and device times (YcStats.gpuMs: first unsettled wave's start → last one's end) are complete after that. */
int yc_render_wave_async(yc_ctx* ctx, YcRect pixels, uint32_t sampleOffset, uint32_t waveSamples,
                         uint32_t takenBefore);
int yc_wave_sync(yc_ctx* ctx);
/* The same wave in two steps, for sample sharding across GPUs (SURVEY §8e alternative B; north_star:
 * "per-GPU ... median-of-means and GMoN accumulation buffers are combined with NCCL"):
 *   yc_accumulate_wave  Integrator::render's sample loop (integrator.cpp:19-24) for this GPU's share of the wave:
 *                       the work is cut into units (estimator bucket b = (index in the wave) % m, pixel class c =
 *                       the c-th of bucketShardCount equal ranges of the frame's pixel list) and the call takes
 *                       the units with (b + c) % bucketShardCount == bucketShard.  Each (bucket, pixel) slot
 *                       receives its samples on one GPU, in sample order (the reference's rounding sequence), the
 *                       others stay zero, so the bucket buffers of all shards add up exactly (bitwise, as 32-bit
 *                       integers).  bucketShardCount = 1 takes every sample.
 *   yc_bucket_device_ptrs  the accumulation buffer, for the caller's NCCL all-reduce(sum) as int32:
 *                       `planes` planes of `planePixels` float4 {sum r, g, b, count (uint32 bits)}.
 *   yc_wave_buckets     how many of those planes (the first m) a wave of `waveSamples` samples uses
 *                       (GMoN / MoN: m = min(15, max(1, 1 + 2 * ((n - 5) / 10))), estimator.hpp:94-141; Mean: 1).
 *   yc_finalize_wave    Estimator::getValue per pixel + finishTile's blend and tonemap
 *                       (estimator.hpp:23-141, tile-renderer.hpp:220-239); clears the buckets. */
int yc_accumulate_wave(yc_ctx* ctx, YcRect pixels, uint32_t sampleOffset, uint32_t waveSamples,
                       uint32_t bucketShard, uint32_t bucketShardCount);
int yc_bucket_device_ptrs(yc_ctx* ctx, void** buckets, size_t* bytes, uint32_t* planes, size_t* planePixels);
int yc_wave_buckets(yc_ctx* ctx, uint32_t waveSamples, uint32_t* m);
int yc_finalize_wave(yc_ctx* ctx, YcRect pixels, uint32_t waveSamples, uint32_t takenBefore);
/* Copies the frames to host (either pointer may be NULL).  width·height·V·4 floats each (V views, yc_set_cameras).
 * Replaces reading Renderer::m_buffer (RenderData::buffer, renderer.hpp:22-28). */
int yc_resolve(yc_ctx* ctx, float* hdrRGBA, float* ldrRGBA, YcStats* stats);
/* First-hit AOVs: guide buffers for a denoiser, collected while the frame renders (no extra ray).
 * For each pixel, over the S samples accumulated since yc_begin_frame: H of them are samples whose camera ray hit a
 * surface at bounce 0 (hitB >= 0). These are the hits after alpha testing, i.e. the surface the integrator shades.
 *   albedo RGBA:
 *     rgb = Σ over hit samples of the evaluated base colour (MatEval::base: YcMaterial::base × base texture) / S;
 *     a = H / S (coverage).
 *   normalDepth RGBA:
 *     xyz = Σ over hit samples of the world-space shading normal (SurfRecord::n, which equals YcHit::n; not flipped
 *           toward the camera, not renormalised after averaging) / S;
 *     w = Σ t over hit samples / H. Camera rays have unit direction (camera.cuh:51), so t is the distance from the
 *         ray's lens origin.
 * Misses contribute 0. Where S = 0 everything is 0, and where H = 0, w is 0. Exposure and background do not apply.
 * Sums are float32, start at +0.0, and add one sample at a time. The order is call order, then sample order within a
 * call, which is the order AccumulateK already uses. The final division is IEEE / (__fdiv_rn on the device). This makes
 * the buffers reproducible by a numpy loop.
 *
 *   yc_enable_aovs     switches the collection on (or off) for the frames that follow: valid before yc_begin_frame or
 *                      before the frame's first wave, YC_ERR_STATE later; YC_ERR_UNSUPPORTED with
 *                      YC_INTEGRATOR_NAIVE.  The first enable allocates 32 bytes per path in flight (twice, per lane:
 *                      512 MB at the default capacity) and four float4 and one uint32 per texel of the frame.
 *                      yc_accumulate_wave with bucketShardCount > 1 returns YC_ERR_UNSUPPORTED while AOVs are on.
 *   yc_resolve_aovs    copies both planes (width·height·V·4 floats each; either pointer may be NULL); YC_ERR_STATE
 *                      when AOVs are not enabled.
 *   yc_comm_reduce_aovs  tile sharding, collective: combines every participant's planes into the root's, out of place
 *                      (repeated calls count nothing twice); yc_resolve_aovs_combined copies them out on the root. */
int yc_enable_aovs(yc_ctx* ctx, int enable);
int yc_resolve_aovs(yc_ctx* ctx, float* albedoRGBA, float* normalDepthRGBA);
/* Adaptive sampling: a pixel stops taking samples once its noise estimate, and its neighbours', is below a threshold.
 * Per texel, over the samples it has taken since yc_begin_frame:
 *   S  the samples taken in the wave calls that finalized (an aborted call adds none).
 *   n, s1, s2  over the samples the frame's estimator accepts (GMoN: no negative channel; all: no NaN), with Y = luma
 *      (0.2126 r + 0.7152 g + 0.0722 b, in that order) of the exposure-scaled sample the estimator adds: n is their
 *      count, s1 = ΣY and s2 = Σ(Y·Y), float32 from +0, one sample at a time in sample order (AccumulateK's order).
 *   e  after each finalizing wave call (yc_render_wave[_async]), for every pixel of the call still sampling:
 *      +inf if n < 2; otherwise mean = s1 / n, var = (s2 - s1·mean) / (n - 1), var = 0 unless var > 0, and
 *      e = sqrt(var / n) / (mean > lumaFloor ? mean : lumaFloor).  float32, IEEE division and sqrt, no contraction.
 *      Texels never sampled read e = +inf.
 *   Stop rule, after e: a pixel of the call stops when S >= minSamples and every e of its neighbourhood is < threshold.
 *      The neighbourhood is the pixel and its 8 neighbours that lie in the same view and the same reference tile (so the
 *      decision never needs another shard's pixels and is the same for any shard count).  The comparison is strict:
 *      NaN never stops a pixel, threshold = 0 stops none.
 *   A stopped pixel takes no further sample in the frame: every later wave call, whatever its rectangle, skips it, so
 *   its HDR, LDR, AOV sums and S keep the values of the wave it stopped at — bit for bit the frame the same calls give
 *   without adaptive sampling after that wave.  Pixels still sampling get exactly the bits of that render.
 *   Scheduling: a wave call starts only after the previous one's stop test (the host reads the count of pixels still
 *   sampling to cut the wave), so yc_render_wave_async overlaps less; the results are the same bits.
 *   Abort: S and e keep describing the waves finished before an aborted call; its partly added n, s1, s2 stay until the
 *   next yc_begin_frame, like the half-filled estimator buckets (yc_set_abort_flag).
 *
 *   yc_set_adaptive    params (NULL: off) for the frames that follow: valid before yc_begin_frame or before the frame's
 *                      first wave, YC_ERR_STATE later; YC_ERR_INVALID for a threshold that is negative or not finite or
 *                      a lumaFloor that is not finite and > 0.  Per texel of the frame it allocates 32 bytes (40 once
 *                      yc_comm_reduce_adaptive ran), per pixel of the shard 32.  While it is on, yc_accumulate_wave
 *                      and yc_finalize_wave return YC_ERR_UNSUPPORTED (bucket sharding would split a pixel's samples
 *                      over the participants, and the sums would lose their order).
 *   yc_resolve_adaptive  copies the planes samples (S, uint32) and error (e, float32), width·height·V texels each, and
 *                      *activePixels, the pixels of this context still sampling (any pointer may be NULL).  YC_ERR_STATE
 *                      when adaptive sampling is off for the frame.
 *   yc_comm_reduce_adaptive  tile sharding, collective: combines every participant's planes into the root's, as
 *                      yc_comm_reduce_aovs does (bit-identical to one context's planes); yc_resolve_adaptive_combined
 *                      copies them out on the root. */
int yc_set_adaptive(yc_ctx* ctx, const YcAdaptive* params);
int yc_resolve_adaptive(yc_ctx* ctx, uint32_t* samples, float* error, uint64_t* activePixels);
/* Device pointers of the frames (for NCCL reductions by the caller); *bytes = width·height·V·4 floats. */
int yc_frame_device_ptrs(yc_ctx* ctx, void** hdr, void** ldr, size_t* bytes);
/* Re-run the tonemap over the whole HDR frame (after a cross-GPU sum). */
int yc_retonemap(yc_ctx* ctx);
/* Bit 0: record per-launch CUDA-event time of the extend kernel into YcStats (bench roofline).
 * Bit 1: run the counting builds of extend / shadow so YcStats.boxTests / triTests accumulate
 * (reference-traversal work; the counting builds do not park leaves speculatively).
 * Bit 2: record per-bounce CUDA-event time of the surface-shading kernels and the hits they shaded.
 * Bit 3: issue a wave's chunks one after the other on one stream instead of two chunks in flight, so that the event
 * times of bits 0 and 2 are the launches' own durations (slower waves; results unchanged). */
int yc_set_profiling(yc_ctx* ctx, int flags);
/* Ray-level parity hook: RayIntegrator::testNode on caller rays (ray-integrator.cpp:20-54). */
int yc_trace(yc_ctx* ctx, const YcRay* rays, size_t n, int mode, YcHit* hits, YcStats* stats);
/* Same with rays already resident on the device; hitsDev receives n compact 20-byte records
 * {f32 t, u, v; u32 prim; i32 node | backSide << 30 (-1 = miss)}.
 * `repeat` back-to-back launches timed with CUDA events → *ms is the average per launch. */
int yc_trace_device(yc_ctx* ctx, const void* raysDev, size_t n, int mode, void* hitsDev, int repeat,
                    float* ms);
int yc_device_alloc(yc_ctx* ctx, size_t bytes, void** out);
int yc_device_free(yc_ctx* ctx, void* p);
/* Page-locked host memory for frame read-back / ray upload at full PCIe rate (optional: every entry
 * point also accepts ordinary pageable memory). */
int yc_host_alloc(yc_ctx* ctx, size_t bytes, void** out);
int yc_host_free(yc_ctx* ctx, void* p);
int yc_memcpy_h2d(yc_ctx* ctx, void* dst, const void* src, size_t bytes);
int yc_memcpy_d2h(yc_ctx* ctx, void* dst, const void* src, size_t bytes);
/* Primary rays exactly as RayIntegrator::sample generates them (ray-integrator.cpp:11-18),
 * written to a device YcRay array of width*height*V*spp entries (sample-major; within a sample, the shard's pixel list
 * order: view after view). */
int yc_generate_primary_rays(yc_ctx* ctx, uint32_t sampleOffset, uint32_t spp, void* raysDev);
int yc_synchronize(yc_ctx* ctx);
/* Renderer::abort (src/core/renderer.hpp:77-83, tile-renderer.hpp:40-63): `flag` is polled between chunks and between
 * bounces of a wave; once it is non-zero the call in progress stops issuing work and returns YC_ERR_ABORTED (the
 * frame keeps the waves finished before; the next yc_begin_frame clears the half-filled accumulation buffers).
 * NULL removes the flag. */
int yc_set_abort_flag(yc_ctx* ctx, const volatile int32_t* flag);

/* --- device layer: combining accumulation buffers across GPUs (north_star: "per-GPU radiance, median-of-means and
 * GMoN accumulation buffers are combined with NCCL over NVLink") ------------------------------------------------
 * A context joins a communicator of `world` participants, one per GPU:
 *   yc_comm_init_all     one process, n contexts on n GPUs (ncclCommInitAll); calls below come from one thread per context
 *   yc_comm_init_rank    one process per GPU (torchrun): rank 0 makes an id with yc_comm_unique_id and hands it to the
 *                        others by any control-plane means (ncclCommInitRank)
 *   yc_comm_init_custom  the caller's own sum collective instead of NCCL (MPI, gloo, a test double): fn(buf, count,
 *                        dtype, root, user) sums `count` elements of dtype (0 f32, 1 i32, 2 u64) in place over all
 *                        participants, into `root` only if root >= 0; `buf` is a DEVICE pointer in the CUDA build
 * NCCL is loaded at the first of these calls (libnccl.so.2 through dlopen: single-GPU users need none). */
#define YC_COMM_ID_BYTES 128
typedef int (*yc_collective_fn)(void* buf, size_t count, int dtype, int root, void* user);
int yc_comm_unique_id(void* id128);
int yc_comm_init_rank(yc_ctx* ctx, int rank, int world, const void* id128);
int yc_comm_init_all(yc_ctx** ctxs, int n);
int yc_comm_init_custom(yc_ctx* ctx, int rank, int world, yc_collective_fn fn, void* user);
int yc_comm_destroy(yc_ctx* ctx);
/* Tile sharding (YcFrameDesc.shardIndex / shardCount): every participant's HDR and LDR frames hold its own tiles and
 * zeros elsewhere; their combination — bit-identical to one GPU's frame — lands in `root`'s combined frames, which
 * yc_resolve_combined copies out on the root (the participants' own frames keep blending their tiles wave after wave).
 * Collective: every participant calls it after the wave.  Where all participants can address the root GPU's memory
 * (NVLink peer access — the devices of one process, or one process per GPU through an exported allocation) the
 * finalize kernel has already stored each finished pixel into the root's frame, and this call is a barrier at most
 * (none if yc_comm_sum_u64 ran since the wave); otherwise the frames are summed into the root (ncclReduce / the
 * caller's collective).  yc_comm_frames_direct reports which (after the first yc_comm_reduce_frames of a frame size). */
int yc_comm_reduce_frames(yc_ctx* ctx, int root);
/* Behind yc_render_wave_async: with direct delivery over NCCL the wave's barrier is enqueued after its finalize kernel
 * and not waited for (otherwise the same as yc_comm_reduce_frames, waiting included). */
int yc_comm_reduce_frames_async(yc_ctx* ctx, int root);
int yc_comm_frames_direct(yc_ctx* ctx, int* direct);
/* The root's combined frames: width·height·V·4 floats each (either pointer may be NULL). */
int yc_resolve_combined(yc_ctx* ctx, float* hdrRGBA, float* ldrRGBA);
/* Bucket sharding (yc_accumulate_wave): all-reduce(sum, int32) of the planes a wave of `waveSamples` samples uses. */
int yc_comm_allreduce_buckets(yc_ctx* ctx, uint32_t waveSamples);
/* Tile sharding with AOVs (yc_enable_aovs): see there. */
int yc_comm_reduce_aovs(yc_ctx* ctx, int root);
int yc_resolve_aovs_combined(yc_ctx* ctx, float* albedoRGBA, float* normalDepthRGBA);
/* Tile sharding with adaptive sampling (yc_set_adaptive): see there. */
int yc_comm_reduce_adaptive(yc_ctx* ctx, int root);
int yc_resolve_adaptive_combined(yc_ctx* ctx, uint32_t* samples, float* error);
/* Control values (ray counts, abort votes): in-place sum over all participants. */
int yc_comm_sum_u64(yc_ctx* ctx, uint64_t* values, uint32_t n);
/* The reference's binned-SAH BVH (src/core/bvh.hpp:140-184, 273-347) built on the device, level by level: the same
 * tree, the same node numbering and the same triangle order as the host builder — and the reference — produce.
 * `nodes` (capacity 2 * nTris + 2) receives the reference's BVHNode array (bvh.hpp:21-33): span == 0 marks an inner node
 * whose children are leftFirst and leftFirst + 1, otherwise a leaf over indices[leftFirst .. leftFirst + span).
 * `faces4`: 4 words per triangle (3 vertex indices, 1 ignored).  Vertex positions must be finite. */
typedef struct YcBuildNode {
  float mn[3], mx[3];
  uint32_t leftFirst, span;
} YcBuildNode;
int yc_build_bvh_sah(int device, const float* positions, size_t nVerts, const uint32_t* faces4, size_t nTris,
                     YcBuildNode* nodes, uint32_t* nNodes, uint32_t* indices, uint32_t* levels);
const char* yc_build_last_error(void);
/* Function-level hooks used by the parity tests (device evaluations of the restated math). */
int yc_kat(yc_ctx* ctx, const char* kind, const void* in, size_t inBytes, void* out, size_t outBytes);

/* --- host layer: scene -------------------------------------------------------------- */
typedef struct ys_scene ys_scene;

/* Loads a ".ysc" scene description (yart_b200/host/scene_desc.hpp) and builds it through the
 * same steps gltf::load performs on the reference API (materials, meshes + SAH BVH, node tree,
 * lights).  Stands in for `gltf::load(path)` (src/gltf/gltf.cpp:319-358). */
int ys_scene_load(const char* path, ys_scene** out);
/* The same with Mesh::BVHType chosen (src/core/mesh.hpp:17): YS_BVH_SAH = SahBVH (what the reference instantiates,
 * bvh.hpp:266-347), YS_BVH_MEDIAN_SPLIT = MedianSplitBVH (bvh.hpp:237-264, its baseline builder). */
#define YS_BVH_SAH 0
#define YS_BVH_MEDIAN_SPLIT 1
/* Where SahBVH is built.  YS_BVH_SAH picks by itself: meshes of at least 32768 triangles with finite vertex data on
 * the GPU (yc_build_bvh_sah, on the device ys_set_build_device chose) when there is one, everything else — and
 * everything after a failure of the device build, or with YART_B200_BVH_DEVICE=0 in the environment — on the host cores
 * (host/bvh_build.hpp, multithreaded).  Same tree either way, node for node. */
#define YS_BVH_SAH_DEVICE 2 /* always through yc_build_bvh_sah (an error if that fails) */
#define YS_BVH_SAH_HOST 3   /* always on the host cores */
int ys_scene_load_bvh(const char* path, uint32_t bvhKind, ys_scene** out);
/* Environment map handed to the GLB entry points: main.cpp:81-84 adds an ImageInfiniteLight(sceneRadius,
 * &hdri) after gltf::load.  rgb = width*height*3 floats in octahedral layout; transform row-major 4x4. */
typedef struct YsEnvLight {
  uint32_t width, height;
  const float* rgb;
  float sceneRadius;
  int32_t hasTransform;
  float transform[16];
} YsEnvLight;
/* gltf::load(path) for binary glTF (src/gltf/gltf.cpp:319-358), from scratch (fastgltf is not vendored in the
 * reference): materials with the KHR extensions the reference enables, merged meshes, TRS node tree, one
 * AreaLight per emissive triangle.  env may be NULL. */
int ys_scene_load_glb(const char* path, const YsEnvLight* env, ys_scene** out);
/* Same, written out as a .ysc description (so the identical scene can be fed to the oracle driver). */
int ys_glb_convert(const char* glbPath, const char* yscPath, const YsEnvLight* env);
/* loadTexture<C> (src/core/texture.hpp:62-90) on an in-memory PNG or JPEG (what stbi_load_from_memory decodes there;
 * host/images.cpp): decode to RGBA8, pick `channels`, sRGB → gamma-2 8-bit.  out may be NULL to query the size. */
int ys_decode_texture(const void* png, size_t len, uint32_t type, uint32_t nChannels, const int32_t* channels,
                      uint8_t* out, size_t outBytes, uint32_t* width, uint32_t* height);
/* loadTextureHDR (src/core/texture.cpp:21-35 = stbi_loadf on a Radiance .hdr): width*height*3 floats.  rgb may be NULL
 * to query the size.  The result is what YsEnvLight::rgb takes (main.cpp:81-84). */
int ys_load_hdr(const char* path, uint32_t* width, uint32_t* height, float* rgb, size_t rgbFloats);
/* output::writePPM (src/output/ppm.cpp:6-21) on an RGBA float frame. */
int ys_write_ppm(const char* path, const float* rgba, uint32_t width, uint32_t height);
/* A float image as a Portable Float Map (what denoiser command-line tools read): `channels` 3 ("PF") or 1 ("Pf"), the
 * first floats of each pixel of `strideFloats` floats (the depth of a normalDepth plane: data = plane + 3, stride 4,
 * channels 1); little-endian (scale -1.0), rows bottom to top as the format requires. */
int ys_write_pfm(const char* path, const float* data, uint32_t width, uint32_t height, uint32_t strideFloats, uint32_t channels);
void ys_scene_destroy(ys_scene* s);
const char* ys_last_error(void);
/* Flattened view (valid until ys_scene_destroy). */
const YcScene* ys_scene_flat(const ys_scene* s);
/* The library's data tables for YcScene::lutTables (the values of the reference's src/bsdf/luts.hpp, 14112 floats). */
const float* ys_lut_tables(size_t* count);
double ys_scene_build_ms(const ys_scene* s);
uint32_t ys_scene_device_builds(const ys_scene* s); /* meshes whose SAH BVH was built on the GPU */
/* BVH of mesh `mesh` in the REFERENCE's node numbering/layout (for builder parity tests):
 * nodes = nNodes × {min[3] max[3] leftFirst span} (32 B), indices = nTris × u32. */
/* Device the SAH builds of later scene loads run on (default 0; -1: host builds only). */
int ys_set_build_device(int device);
int ys_scene_bvh(const ys_scene* s, uint32_t mesh, const void** nodes, uint32_t* nNodes,
                 const uint32_t** indices, uint32_t* nTris);

/* Camera(imageSize, focalLength, fNumber) + moveAndLookAt(position, target, up)
 * (src/core/camera.hpp:77-136); up = (0,0,0) keeps the default +Y. */
int ys_camera_make(uint32_t width, uint32_t height, float focalLength, float fNumber,
                   const float position[3], const float target[3], const float up[3],
                   float exposure, uint32_t apertureSides, YcCamera* out);

/* --- host layer: renderer ----------------------------------------------------------- */
/* Mirror of cpu::TileRenderer's public knobs (tile-renderer.hpp:27-32) + Renderer fields. */
typedef struct YrSettings {
  uint32_t width, height;
  uint32_t samples, firstWaveSamples, maxWaveSamples, tileSize;
  uint32_t maxDepth;
  float background[3];
  uint32_t tonemap;   /* YC_TONEMAP_* (tonemapper == nullptr ↔ NONE) */
  uint32_t estimator; /* YC_ESTIMATOR_* */
  uint32_t shardIndex, shardCount;
  int32_t device;
  uint32_t integrator; /* YC_INTEGRATOR_* */
  uint32_t scrambler;  /* YC_SCRAMBLER_* */
  uint32_t sampler;    /* YC_SAMPLER_* */
  uint32_t traversal;  /* YC_TRAVERSAL_* */
  uint32_t sharding;   /* YR_SHARD_*: how yr_create_multi / yr_create_dist split a wave across GPUs */
} YrSettings;

#define YR_SHARD_TILES 0   /* tile k of the reference's tile list (tile-renderer.hpp:127-144) → GPU k mod G; frames reduced to rank 0 */
#define YR_SHARD_BUCKETS 1 /* every GPU holds the frame and takes (estimator bucket, pixel class) units of each wave; the
                              GMoN accumulation buffers are all-reduced per wave; every GPU ends up with the frame */

typedef struct YrRenderData {  /* Renderer::RenderData (renderer.hpp:22-28) */
  uint64_t samplesTaken, totalSamples, totalRays;
  double totalTimeMs;
} YrRenderData;

typedef struct YrWaveData {    /* Renderer::WaveData (renderer.hpp:33-38) */
  uint64_t wave, waveSamples, rays;
  double timeMs;
} YrWaveData;

typedef struct YrTileData {    /* Renderer::TileData (renderer.hpp:43-50) */
  uint32_t x, y, w, h;
  uint64_t index, total, rays;
  double timeMs;
} YrTileData;

typedef void (*yr_wave_callback)(const YrRenderData*, const YrWaveData*, void* user);   /* onRenderWaveComplete */
typedef void (*yr_tile_callback)(const YrRenderData*, const YrTileData*, void* user);   /* onRenderTileComplete */
typedef void (*yr_done_callback)(const YrRenderData*, int aborted, void* user);         /* onRenderComplete / onRenderAborted */

typedef struct yr_renderer yr_renderer;
int yr_create(const YrSettings* settings, const ys_scene* scene, const YcCamera* camera, yr_renderer** out);
/* The same on a caller-flattened scene (what a `yart::Renderer` subclass holding `const Scene* scene`,
 * renderer.hpp:53, passes: integration/wavefront-renderer.hpp).  The arrays must outlive the renderer. */
int yr_create_flat(const YrSettings* settings, const YcScene* scene, const YcCamera* camera, yr_renderer** out);
/* One renderer over several GPUs of this process (scene replicated, one driver thread per GPU, NCCL inside):
 * render / abort / wait / callbacks / read are unchanged and the frame is bit-identical to one GPU's.
 * Replaces TileRenderer's worker threads (tile-renderer.hpp:150-197) at the scale of a box. */
int yr_create_multi(const YrSettings* settings, const ys_scene* scene, const YcCamera* camera, const int* devices,
                    uint32_t nDevices, yr_renderer** out);
int yr_create_multi_flat(const YrSettings* settings, const YcScene* scene, const YcCamera* camera, const int* devices,
                         uint32_t nDevices, yr_renderer** out);
/* The same with one process per GPU (torchrun): settings->device is this process's GPU, `commId` the bytes rank 0 got
 * from yc_comm_unique_id.  Rank 0 receives the frame (tile sharding) or every rank does (bucket sharding); ray counts
 * in YrRenderData / YrWaveData are whole-job figures on every rank. */
int yr_create_dist(const YrSettings* settings, const ys_scene* scene, const YcCamera* camera, int rank, int world,
                   const void* commId, yr_renderer** out);
int yr_create_dist_custom(const YrSettings* settings, const ys_scene* scene, const YcCamera* camera, int rank, int world,
                          yc_collective_fn fn, void* user, yr_renderer** out);
void yr_destroy(yr_renderer* r);
int yr_set_wave_callback(yr_renderer* r, yr_wave_callback cb, void* user);
int yr_set_tile_callback(yr_renderer* r, yr_tile_callback cb, void* user);
int yr_set_done_callback(yr_renderer* r, yr_done_callback cb, void* user);
/* Host frame (width*height*V*4 floats, V views of yr_set_cameras stacked by rows) that receives the tonemapped frame — the HDR one when tonemap is NONE, like
 * Renderer::m_buffer (tile-renderer.hpp:238) — after every wave, before the callbacks fire. */
int yr_set_frame_target(yr_renderer* r, float* ldrRGBA);
int yr_set_camera(yr_renderer* r, const YcCamera* camera); /* the camera moved between renders */
/* n views of the scene per render (yc_set_cameras: 1 <= n <= 65535, stacked by rows, each bit-identical to a render of
 * its camera alone).  Like yr_set_camera it waits for a render in progress and applies to the next one; the count may
 * change between renders.  Frames, AOV planes, the frame target and the PPM are width x (height·n); the tile callback
 * reports every tile of every view per wave (stacked x, y, w, h; index over all n views, total = n x tiles per view). */
int yr_set_cameras(yr_renderer* r, const YcCamera* cameras, uint32_t n);
int yr_render(yr_renderer* r);     /* Renderer::render(): asynchronous */
int yr_abort(yr_renderer* r);      /* Renderer::abort(): returns at once, the render stops at its next chunk / bounce */
int yr_wait(yr_renderer* r);       /* Renderer::wait() */
int yr_render_sync(yr_renderer* r, YrRenderData* out); /* Renderer::renderSync() */
/* Result buffers: LDR (what Renderer::m_buffer holds) and HDR accumulation. */
int yr_read(yr_renderer* r, float* hdrRGBA, float* ldrRGBA, YcStats* stats);
/* First-hit AOVs of the renders that follow (yc_enable_aovs; YC_ERR_UNSUPPORTED for the naive integrator and for
 * YR_SHARD_BUCKETS over more than one participant, YC_ERR_STATE while a render runs). */
int yr_enable_aovs(yr_renderer* r, int enable);
/* The AOV planes of the last render (width*height*V*4 floats each, either pointer may be NULL), valid once it has returned
 * (yr_render_sync / yr_wait) and YC_ERR_STATE while one runs.  Tile sharding: the combined planes, on the root; other
 * ranks' buffers are left untouched, as with yr_read. */
int yr_read_aovs(yr_renderer* r, float* albedoRGBA, float* normalDepthRGBA);
/* Adaptive sampling for the renders that follow (yc_set_adaptive; NULL: off).  YC_ERR_INVALID for bad parameters,
 * YC_ERR_UNSUPPORTED for YR_SHARD_BUCKETS over more than one participant, YC_ERR_STATE while a render runs.  A render
 * ends early, as a normal completion (done callback with aborted = 0), after the first wave that leaves no pixel sampling
 * on any participant; YrRenderData.samplesTaken is then the schedule's samples up to that wave.  The wave and tile
 * callbacks and the frame target fire for every wave that ran. */
int yr_set_adaptive(yr_renderer* r, const YcAdaptive* params);
/* The samples / error planes of the last render (width*height*V texels each, either pointer may be NULL), valid once it
 * has returned.  Tile sharding: the combined planes, on the root (combined once per render, aborted renders included). */
int yr_read_adaptive(yr_renderer* r, uint32_t* samples, float* error);
/* writePPM(out, renderer buffer): the tonemapped frame as a binary PPM (frontend main.cpp writes out.ppm); width x
 * (height·V) with several views. */
int yr_write_ppm(yr_renderer* r, const char* path);
yc_ctx* yr_context(yr_renderer* r);
const char* yr_last_error(const yr_renderer* r);

#ifdef __cplusplus
}
#endif
#endif /* YART_CUDA_H */
