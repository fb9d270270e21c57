// core_internal.h — host-side state of a pt_context (not part of the C ABI).
#pragma once
#include <cuda_runtime.h>

#include <algorithm>
#include <string>
#include <vector>

#include "../../include/pt_core.h"
#include "scene.cuh"

#define PT_CUDA_CHECK(ctx, expr)                                                                                      \
    do                                                                                                                \
    {                                                                                                                 \
        cudaError_t err__ = (expr);                                                                                   \
        if (err__ != cudaSuccess)                                                                                     \
            return pt::fail(ctx, err__ == cudaErrorMemoryAllocation ? PT_ERR_OUT_OF_MEMORY : PT_ERR_CUDA, #expr,      \
                            cudaGetErrorString(err__));                                                               \
    } while (0)

namespace pt
{

// device counters, one cache line each would be overkill: they are touched once per block
struct DeviceCounters
{
    unsigned long long raysClosest, raysShadow, samples, hits, boxClosest, triClosest, alphaClosest, boxShadow, triShadow,
        alphaShadow, texels, restarts;
    unsigned long long visitHist[8], warpIters, warpDrainIters, maxWarpDrainIters; // diagnostics (stats runs)
};

// wavefront queue bookkeeping living in device memory
struct QueueCounts
{
    uint32_t cont[2];  // double-buffered queue sizes: continuing paths ...
    uint32_t regen[2]; // ... and ended paths whose slot takes the next work item inside k_extend
    uint32_t hit;      // slots whose closest-hit query hit (input of k_shade)
    uint32_t pad2[2];
    uint32_t shadow;
    uint32_t extendWork; // ray-queue positions handed out to the persistent warps of k_extend ...
    uint32_t shadowWork; // ... and k_shadow
    uint32_t pad;
};

// Path state: one 256-byte record per slot of the pool (a slot carries one path = one work item
// at a time).  Array-of-structures ON PURPOSE: every kernel reaches the state through a queue of
// slot indices, i.e. in random order, so what counts is how many DRAM pages / L2 lines one path
// touches, not coalescing across neighbouring threads.  A structure-of-arrays layout (the first
// version) spread one path over 13 lines in 13 pages and ran at the random-access DRAM rate.
struct __align__(128) PathRecord
{
    // line A — the bounce state (k_extend reads rayO/rayD, k_shade reads and rewrites all of it)
    float4 rayO;  // origin.xyz, maxRoughness
    float4 rayD;  // direction.xyz, rng (bits)
    float4 thr;   // throughput.xyz, bits: bounce count | NaN/Inf restarts of the sample << 8
    float4 rad;   // radiance.xyz, work item (bits): round-relative sample * pixelCount + pixel-list index
    float4 diff0; // rxOrigin.xyz, rxDirection.x
    float4 diff1; // rxDirection.yz, ryOrigin.xy
    float4 diff2; // ryOrigin.z, ryDirection.xyz
    float4 hit;   // tri (bits), t, b1, b2
    // line B — the shadow ray and the decal record
    float4 shO;   // shadow origin.xyz, tmax
    float4 shD;   // shadow direction.xyz, -
    float4 shC;   // contribution.xyz (throughput * DirectLight / pdf), -
    float4 decal; // rgb, dist (scenes with alpha-tested geometry)
    float decalA;
    uint32_t pad[3]; // pad[0]: bsdf.Pdf of the previous bounce (k_shade<A, S, true>, emissive-MIS light sampling)
    float4 spare[3];
};
static_assert(sizeof(PathRecord) == 256, "PathRecord must be two 128-byte lines");

struct PathState
{
    PathRecord *rec;
    uint32_t *contQ[2];  // active slots with a continuing path, double buffered
    uint32_t *regenQ[2]; // slots whose path has ended (| PT_REGEN, | PT_REGEN_MISS if it left the scene), double buffered
    uint32_t *hitQ;      // slots to shade (k_extend order)
    uint32_t *hitKey;    // sort key of hitQ[i]: leaf-order triangle index >> hitKeyShift (0xffffffff = unused)
    uint32_t *hitQSorted, *hitKeySorted; // after the radix sort: coherent warps for k_shade
    uint32_t *shadowQueue;
};

#define PT_MAX_POOLS 8

// Emissive triangles for next-event estimation (emitters.cu; PT_LIGHT_SAMPLING_EMISSIVE_MIS only).  Emitter k of the table
// is flat triangle flatIds[k]; it is drawn with probability weight[k] / sum(weight) through the alias table.
struct EmitterTable
{
    const float4 *rec;          // [count][4]: p0.xyz, p1.x | p1.yz, p2.xy | p2.z, uv0, uv1.x | uv1.y, uv2, material id (bits)
    const uint2 *alias;         // [count]: (threshold of the 32-bit fraction, alias index)
    const float *emitterPdf;    // [count]: P(select) / area of emitter k
    const float *pdfOverArea;   // [flat triangles]: the same by flat id, 0 for triangles that are never sampled
    uint32_t count;
    float pEmitter;             // probability of the emitter branch of a light sample
};

// Adaptive sampling (DESIGN.md §3i): Welford statistics of the luminance of a pixel's samples, in sample order
struct __align__(16) AdaptivePixel
{
    uint32_t count; // samples the pixel has
    float mean, m2;
    uint32_t pad;
};

// what k_adaptive_blocks / k_adaptive_select / k_adaptive_scatter report to the host after an evaluation
struct AdaptiveSummary
{
    uint32_t n;            // smallest count among the active blocks (0xffffffff: none is active)
    uint32_t next;         // next larger count among them (0xffffffff: none)
    uint32_t pixels;       // A: pixels of the active blocks at count n = the pass's pixel list
    uint32_t minCount, maxCount;
    uint32_t unconverged;  // pixels of blocks at or above max_samples that miss the threshold
    uint32_t pad[2];
};

// host copy of the tables instances are flattened from (kept for pt_scene_update)
struct SceneTopology
{
    std::vector<pt_instance> instances;
    std::vector<pt_model> models;
    std::vector<pt_mesh_record> meshRecords;
    std::vector<pt_geometry> geometries;
    std::vector<float> transforms; // 12 per mesh transform
    uint64_t vertexCount = 0, indexCount = 0;
    uint32_t materialCount[3] = { 0, 0, 0 };
    // skeletal animation: animated geometries address the animated buffers, which the core keeps
    // BEHIND the static ones (skinned vertices at vertexCount + i, animated indices at indexCount + i)
    std::vector<uint32_t> geometryIsAnimated;
    uint64_t animatedVertexCount = 0, animatedIndexCount = 0;
    uint32_t boneCount = 0;
};

struct Context
{
    int device = 0;
    int smCount = 0;
    uint32_t traceBlocksPerSM = 0; // 0 = occupancy query; PT_TRACE_BLOCKS overrides (tuning)
    cudaStream_t stream = nullptr;
    cudaMemPool_t memPool = nullptr; // private stream-ordered pool: nothing of the host application's default pool is touched
    std::string lastError;

    // scene
    bool hasScene = false;
    DeviceScene scene = {};
    std::vector<void *> sceneAllocs; // everything cudaMalloc'ed for the scene ...
    std::vector<void *> accelAllocs; // ... except the triangle streams + BVH, which pt_scene_update rebuilds
    SceneTopology topo;
    const float *dVertices = nullptr;    // the reference's vertex buffer, 14 floats per vertex (+ the skinned vertices)
    const uint32_t *dIndices = nullptr;
    const float *dAnimatedVertices = nullptr; // Shaders::AnimatedVertex, 22 words per vertex (bind pose)
    float *dBones = nullptr;                  // per bone: 12 floats of the matrix + 9 of its normal matrix
    LightBlock hostLights = {};
    uint32_t sceneUpdates = 0;
    std::vector<DevTexture> hostTextures;
    uint64_t texelArenaBytes = 0;
    uint64_t nodeCount = 0, bvhBytes = 0;
    float bvhBuildMs = 0, sceneUploadMs = 0;
    uint32_t bvhBuilder = 1;  // 1 = PLOC (default), 0 = LBVH; PT_BVH / tuning key "bvh_builder"
    uint32_t plocRadius = 8;  // PLOC search window on either side; PT_PLOC_RADIUS / "ploc_radius"
    uint32_t bvhBuildPasses = 0;
    // TextureUploader's limits: textures beyond maxTextureSize (MaxTextureDataSize = 4096, always) or beyond the per-texture share
    // of textureBudgetBytes (0 = ForceFullTextureSize, the default on a 180 GB device) are scaled down at upload
    uint32_t maxTextureSize = 4096;
    uint64_t textureBudgetBytes = 0;
    uint32_t textureBudgetCount = 1; // scene textures sharing the budget
    uint32_t maxAnisotropy = 1; // sampler state (pt_set_sampler): 1 = isotropic trilinear, 16 = the reference's sampler
    // reference splitting (bvh_build.cu k_split_*): a triangle whose box volume exceeds splitThreshold x the scene volume per
    // primitive enters the BVH as 4^L references; 0 = off.  Tuning key "split_threshold_x100" / PT_SPLIT.
    float splitThreshold = 4.0f;
    uint64_t triangleCount = 0, referenceCount = 0;
    uint32_t bvhMaxDepth = 0; // levels of the wide BVH (the traversal stack holds at most 3 entries per level)

    // light sampling (pt_set_light_sampling) and the emitter table, built at the first render that needs it after the
    // scene, a texture or the sampler changed; nothing of it exists in the default mode
    uint32_t lightSampling = PT_LIGHT_SAMPLING_REFERENCE;
    bool emittersValid = false;
    EmitterTable emitters = {};
    std::vector<void *> emitterAllocs;
    std::vector<uint32_t> emitterIds, emitterWeights;
    std::vector<uint2> emitterAlias;
    float emitterBuildMs = 0;

    // target
    uint32_t width = 0, height = 0;
    float4 *accum = nullptr;
    PathState ps = {};
    std::vector<void *> targetAllocs;
    // denoiser buffers (denoise.cu), one target allocation made at the first pt_denoise: guides (albedo, t) and (N, 0), the
    // result, the filter's (N, t) taps, two ping-pong (irradiance, variance) images and the depth gradient
    float4 *denoiseAlbedoT = nullptr, *denoiseNormal = nullptr, *denoised = nullptr, *denoiseNT = nullptr;
    float4 *denoisePing = nullptr, *denoisePong = nullptr;
    float2 *denoiseGrad = nullptr;
    bool denoiseValid = false; // a pt_denoise result exists for the current accumulation
    // temporal denoiser state (temporal.cu, DESIGN §3j), one target allocation made at the first pt_denoise_temporal:
    // two history buffers of (integrated irradiance.rgb, history length n) and (m1, m2) -- one is read while the other is
    // written -- and the previous call's (N, t) taps (t = -1 where the pixel was invalid).  The previous camera is kept
    // here.  It survives pt_render_begin at the same extent; scene and texture uploads and updates clear temporalValid.
    float4 *temporalIrr[2] = {};
    float2 *temporalMoments[2] = {};
    float4 *temporalPrevNT = nullptr;
    uint32_t temporalCurrent = 0; // temporalIrr / temporalMoments[temporalCurrent] hold the history after the last call
    bool temporalValid = false;
    float temporalPrevView[16] = {}, temporalPrevProj[16] = {};
    // what the accumulation holds since the last pt_render_begin: nothing, a uniform render (pt_render_samples /
    // pt_render_frames) or an adaptive one (pt_render_adaptive); the two never mix, so per-pixel counts stay known
    enum class TargetContent { Empty, Uniform, Adaptive } targetContent = TargetContent::Empty;
    // adaptive sampling (adaptive.cu), one target allocation made at the first pt_render_adaptive: per pixel (count, mean
    // luminance, M2), per 8x4 block three words and the scan's scratch, and the pass summary; the mean image accum / count
    // at the first read
    AdaptivePixel *adaptivePixels = nullptr;
    uint32_t *adaptiveBlocks = nullptr;
    uint32_t *adaptiveCounts = nullptr, *adaptiveOffsets = nullptr; // per block: pixels selected for the pass, their scan
    void *adaptiveScanTemp = nullptr;
    size_t adaptiveScanBytes = 0;
    AdaptiveSummary *adaptiveSummary = nullptr;
    float4 *adaptiveMean = nullptr;
    size_t slotPoolSize = (size_t)1 << 23;     // paths in flight, all pools together (PT_SLOTS)
    size_t sbufBudgetBytes = (size_t)8 << 30;  // sample-buffer budget (PT_SBUF_MB)
    uint32_t slotCapacity = 0; // size of the slot pool
    // pixel list of the current tile set in 8x4-block order (rebuilt only when the tile list changes)
    uint32_t *pixelList = nullptr;
    std::vector<pt_tile> pixelTiles;
    uint32_t pixelCount = 0;
    bool pixelListValid = false;
    // sample buffer of one round: [samples][pixelCount] float4, grown on demand
    float4 *sbuf = nullptr;
    uint64_t sbufCapacity = 0; // float4 entries
    bool collectTraversalStats = false;
    bool kernelTiming = false;

    bool sortHits = true;       // PT_SORT_HITS=0 disables (tuning)
    void *sortTemp = nullptr;   // CUB radix-sort scratch for slotCapacity pairs
    size_t sortTempBytes = 0;

    uint32_t poolCount = 2;     // independent sub-wavefronts (PT_POOLS); 2 measured best once k_extend regenerates paths
    cudaStream_t poolStreams[PT_MAX_POOLS] = {};
    cudaEvent_t evRound = nullptr;

    DeviceCounters *dCounters = nullptr;
    QueueCounts *dQueueCounts = nullptr; // [PT_MAX_POOLS]
    QueueCounts *hQueueCounts = nullptr; // [PT_MAX_POOLS], pinned
    uint32_t *dNextItem = nullptr;       // next work item of the round, shared by the pools
    uint32_t *hNextItem = nullptr;       // pinned
    float *dLut = nullptr;

    // stats of the last call
    pt_stats stats = {};
    cudaEvent_t evStart = nullptr, evStop = nullptr;
};

pt_status fail(Context *ctx, pt_status code, const char *what, const char *detail);

// Every entry point of the C ABI works on the context's device and leaves the caller's current device as it was.
struct DeviceGuard
{
    int previous = -1;
    explicit DeviceGuard(int device)
    {
        if (cudaGetDevice(&previous) != cudaSuccess)
            previous = -1;
        if (previous != device)
            cudaSetDevice(device);
        else
            previous = -1;
    }
    ~DeviceGuard()
    {
        if (previous >= 0)
            cudaSetDevice(previous);
    }
    DeviceGuard(const DeviceGuard &) = delete;
    DeviceGuard &operator=(const DeviceGuard &) = delete;
};

// a CUDA event that is destroyed on every path out of a function
struct ScopedEvent
{
    cudaEvent_t ev = nullptr;
    ScopedEvent() { cudaEventCreate(&ev); }
    ~ScopedEvent()
    {
        if (ev)
            cudaEventDestroy(ev);
    }
    ScopedEvent(const ScopedEvent &) = delete;
    ScopedEvent &operator=(const ScopedEvent &) = delete;
    operator cudaEvent_t() const { return ev; }
};

// stream-ordered allocation from the context's private pool
inline cudaError_t poolAlloc(Context *ctx, void **ptr, size_t bytes, cudaStream_t stream)
{
    return cudaMallocFromPoolAsync(ptr, bytes, ctx->memPool, stream);
}

// traversal-stack overflows since the last call (wavefront.cu); non-zero fails the call that caused them
pt_status checkStackOverflow(Context *ctx, const char *what);

// resident 128-thread blocks per SM the register allocation of the trace kernels (k_extend, k_shadow and their probe
// k_test_trace) must allow (tuned on the B200, see DESIGN.md)
#ifndef PT_TRACE_MIN_BLOCKS
#define PT_TRACE_MIN_BLOCKS 8
#endif
// Grid of a persistent trace launch: exactly as many 128-thread blocks as are resident on the machine (occupancy query
// per instantiation; PT_TRACE_BLOCKS overrides), never more than `items` work items need.
template <class Kernel> uint32_t residentTraceGrid(const Context *ctx, Kernel kernel, uint32_t items)
{
    int perSM = 0;
    if (ctx->traceBlocksPerSM)
        perSM = (int)ctx->traceBlocksPerSM;
    else if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&perSM, kernel, 128, 0) != cudaSuccess || perSM < 1)
        perSM = 4;
    return std::min((items + 127) / 128, (uint32_t)(ctx->smCount * perSM));
}

// bvh_build.cu
pt_status uploadScene(Context *ctx, const pt_scene_desc *desc);
void freeScene(Context *ctx);
pt_status uploadTextureSlot(Context *ctx, uint32_t slot, const pt_texture_desc *tex);
pt_status updateScene(Context *ctx, const pt_scene_update_desc *desc);

// emitters.cu
pt_status buildEmitters(Context *ctx);
void freeEmitters(Context *ctx);

// textures.cu
pt_status createTexture(Context *ctx, const pt_texture_desc &desc, DevTexture &out, void **outAlloc, bool scalable = false);
pt_texture_desc defaultTexture(const uint32_t *rgba, bool srgb);

// wavefront.cu
pt_status allocSortTemp(Context *ctx, size_t slots);
pt_status renderFrames(Context *ctx, const pt_render_params *params, uint32_t firstSample, uint32_t frameCount, uint32_t samplesPerFrame,
                        const pt_tile *tiles, uint32_t tileCount);
// the pieces of renderFrames, in its order: the sample buffer for sampleCount samples of ctx->pixelCount pixels (roundMax =
// samples per round), the counters and the start event, the rounds over ctx->pixelList (k_resolve<adaptive>, which with
// `adaptive` also updates the pixels' statistics), and the stop event, the timing and the stack check
pt_status sizeSampleBuffer(Context *ctx, uint32_t sampleCount, uint32_t &roundMax);
pt_status resetRenderStats(Context *ctx);
pt_status renderRounds(Context *ctx, const pt_render_params *params, uint32_t firstSample, uint32_t sampleCount, uint32_t samplesPerFrame,
                       uint32_t roundMax, bool adaptive);
pt_status finishRender(Context *ctx, const char *what);

// adaptive.cu
pt_status renderAdaptive(Context *ctx, const pt_render_params *params, const pt_adaptive_params *ap, pt_adaptive_info *info);
// accum / count into ctx->adaptiveMean (allocated here), queued on ctx->stream
pt_status adaptiveMeanImage(Context *ctx, const char *what);
pt_status firstHitAov(Context *ctx, const pt_render_params *params, uint32_t width, uint32_t height, pt_hit *out);
pt_status debugRender(Context *ctx, const pt_render_params *params, const pt_debug_params *debug, uint32_t width, uint32_t height,
                      float *out);
pt_status traceClosest(Context *ctx, const pt_ray *rays, uint64_t n, pt_hit *out);
pt_status traceOcclusion(Context *ctx, const pt_ray *rays, uint64_t n, uint8_t *out);
// pt_test_trace: the trace kernels' persistent traversal (or the per-thread one) on host rays
pt_status testTrace(Context *ctx, const pt_ray *rays, uint64_t n, uint32_t flags, uint32_t blocks, pt_hit *out, float *outDecals,
                    uint64_t *outTail);
// k_denoise_guides over the render target's extent, queued on ctx->stream
void launchDenoiseGuides(Context *ctx, const pt_render_params *params, float4 *albedoT, float4 *normal);

// denoise.cu
// src / divisor as in postProcess; src is read after the argument checks, so ctx->accum may still be NULL there.
// checkDenoise / checkPostProcess are those argument checks alone (no device work), run first by both functions
pt_status checkDenoise(Context *ctx, const char *what, const pt_render_params *params, const pt_denoise_params *dn, float divisor,
                       const float *out, size_t outBytes);
pt_status denoise(Context *ctx, const char *what, const pt_render_params *params, const pt_denoise_params *dn, const float4 *src,
                  float divisor, float *out, size_t outBytes);
// the pieces of denoise(), in its order, which pt_denoise_temporal shares: the target's denoiser buffers; the guides and
// k_denoise_prepare (ping = demodulated irradiance); k_denoise_variance of ping into pong; the K a-trous levels starting
// from pong, the last one remodulating into ctx->denoised; and the copy to `out`, the synchronisation, the launch count
// and the stack check
pt_status allocDenoiseBuffers(Context *ctx);
void launchDenoisePrepare(Context *ctx, const pt_render_params *params, const float4 *src, float divisor);
void launchDenoiseVariance(Context *ctx, const pt_denoise_params *dn);
void launchAtrous(Context *ctx, const pt_denoise_params *dn);
pt_status finishDenoise(Context *ctx, const char *what, float *out, uint32_t launches);

// temporal.cu
pt_status denoiseTemporal(Context *ctx, const pt_render_params *params, const pt_denoise_params *dn, const pt_temporal_params *tp,
                          uint32_t totalSamples, float *out, size_t outBytes);
pt_status temporalHistory(Context *ctx, float *outIrradianceN, float *outMoments, size_t pixels);

// postprocess.cu
// src / divisor is the image the chain starts from: the accumulation and its sample count, or the denoised mean and 1
pt_status checkPostProcess(Context *ctx, const char *what, const pt_postprocess_params *params, uint32_t outputFormat, const void *out,
                           size_t outBytes);
pt_status postProcess(Context *ctx, const char *what, const pt_postprocess_params *params, const float4 *src, float divisor,
                      uint32_t outputFormat, void *out, size_t outBytes);

// unit_kernels.cu
void testComposeTransform(const float *meshRows, const float *instanceRows, float P[12], float N[9]);
pt_status testShading(Context *ctx, uint32_t mode, const float *input, float *output, uint32_t count);
pt_status testTexture(Context *ctx, uint32_t slot, const float *in6, float *out4, uint32_t count, int32_t useGrad);
uint32_t testInputStride(uint32_t mode);
uint32_t testOutputStride(uint32_t mode);

} // namespace pt

struct pt_context : pt::Context
{
};
