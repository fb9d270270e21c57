// pt_core.cu — the C ABI of include/pt_core.h: context, render target and dispatch.
#include "core_internal.h"

#include <cmath>
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>

namespace pt
{

static thread_local std::string g_createError;

pt_status fail(Context *ctx, pt_status code, const char *what, const char *detail)
{
    std::string msg = std::string(what) + ": " + detail;
    if (ctx)
        ctx->lastError = msg;
    else
        g_createError = msg;
    return code;
}

static void freeTarget(Context *ctx)
{
    for (void *p : ctx->targetAllocs)
        cudaFree(p);
    ctx->targetAllocs.clear();
    ctx->accum = nullptr;
    ctx->denoiseAlbedoT = ctx->denoiseNormal = ctx->denoised = ctx->denoiseNT = nullptr;
    ctx->denoisePing = ctx->denoisePong = nullptr;
    ctx->denoiseGrad = nullptr;
    ctx->denoiseValid = false;
    ctx->temporalIrr[0] = ctx->temporalIrr[1] = ctx->temporalPrevNT = nullptr;
    ctx->temporalMoments[0] = ctx->temporalMoments[1] = nullptr;
    ctx->temporalCurrent = 0;
    ctx->temporalValid = false;
    ctx->targetContent = Context::TargetContent::Empty;
    ctx->adaptivePixels = nullptr;
    ctx->adaptiveBlocks = nullptr;
    ctx->adaptiveCounts = ctx->adaptiveOffsets = nullptr;
    ctx->adaptiveScanTemp = nullptr;
    ctx->adaptiveScanBytes = 0;
    ctx->adaptiveSummary = nullptr;
    ctx->adaptiveMean = nullptr;
    ctx->ps = PathState {};
    ctx->slotCapacity = 0;
    ctx->pixelList = nullptr;
    ctx->pixelListValid = false;
    ctx->pixelCount = 0;
    cudaFree(ctx->sortTemp);
    ctx->sortTemp = nullptr;
    ctx->sortTempBytes = 0;
    cudaFree(ctx->sbuf);
    ctx->sbuf = nullptr;
    ctx->sbufCapacity = 0;
    ctx->width = ctx->height = 0;
}

template <typename T> static pt_status targetAlloc(Context *ctx, T **ptr, size_t count)
{
    PT_CUDA_CHECK(ctx, cudaMalloc((void **)ptr, std::max<size_t>(count, 1) * sizeof(T)));
    ctx->targetAllocs.push_back(*ptr);
    return PT_OK;
}

} // namespace pt

using namespace pt;

extern "C" {

pt_status pt_context_create(int32_t cuda_device, pt_context **out_ctx)
{
    if (!out_ctx)
        return fail(nullptr, PT_ERR_INVALID_ARGUMENT, "pt_context_create", "out_ctx is NULL");
    *out_ctx = nullptr;
    int count = 0;
    cudaError_t err = cudaGetDeviceCount(&count);
    if (err != cudaSuccess || count == 0)
        return fail(nullptr, PT_ERR_NO_DEVICE, "pt_context_create",
                    err != cudaSuccess ? cudaGetErrorString(err) : "no CUDA device (there is no CPU fallback)");
    if (cuda_device < 0 || cuda_device >= count)
        return fail(nullptr, PT_ERR_INVALID_ARGUMENT, "pt_context_create", "cuda_device out of range");
    cudaDeviceProp prop;
    err = cudaGetDeviceProperties(&prop, cuda_device);
    if (err != cudaSuccess)
        return fail(nullptr, PT_ERR_CUDA, "cudaGetDeviceProperties", cudaGetErrorString(err));
    if (prop.major != 10)
    {
        char buf[128];
        std::snprintf(buf, sizeof(buf), "device %d is sm_%d%d; this library is built for sm_100a only", cuda_device,
                      prop.major, prop.minor);
        return fail(nullptr, PT_ERR_NO_DEVICE, "pt_context_create", buf);
    }
    DeviceGuard guard(cuda_device);

    pt_context *ctx = new pt_context();
    ctx->device = cuda_device;
    ctx->smCount = prop.multiProcessorCount;
    // tuning knobs (not part of the ABI): PT_SLOTS = paths in flight, PT_SBUF_MB = sample-buffer budget
    if (const char *e = std::getenv("PT_SLOTS"))
        ctx->slotPoolSize = std::max<size_t>(1024, std::strtoull(e, nullptr, 10));
    if (const char *e = std::getenv("PT_TRACE_BLOCKS"))
        ctx->traceBlocksPerSM = (uint32_t)std::max(1, std::atoi(e));
    if (const char *e = std::getenv("PT_POOLS"))
        ctx->poolCount = (uint32_t)std::min(PT_MAX_POOLS, std::max(1, std::atoi(e)));
    if (const char *e = std::getenv("PT_SORT_HITS"))
        ctx->sortHits = std::atoi(e) != 0;
    if (const char *e = std::getenv("PT_BVH"))
        ctx->bvhBuilder = std::atoi(e) != 0;
    if (const char *e = std::getenv("PT_PLOC_RADIUS"))
        ctx->plocRadius = (uint32_t)std::max(1, std::atoi(e));
    if (const char *e = std::getenv("PT_SPLIT")) // reference-splitting threshold (0 = off)
        ctx->splitThreshold = (float)std::atof(e);
    if (const char *e = std::getenv("PT_MAX_ANISOTROPY")) // A/B measurements; pt_set_sampler is the API
        ctx->maxAnisotropy = (uint32_t)std::min(16, std::max(1, std::atoi(e)));
    if (const char *e = std::getenv("PT_SBUF_MB"))
        ctx->sbufBudgetBytes = std::max<size_t>(1, std::strtoull(e, nullptr, 10)) << 20;
#define PT_CREATE_CHECK(expr)                                                                                         \
    do                                                                                                                \
    {                                                                                                                 \
        cudaError_t e__ = (expr);                                                                                     \
        if (e__ != cudaSuccess)                                                                                       \
        {                                                                                                             \
            fail(nullptr, PT_ERR_CUDA, #expr, cudaGetErrorString(e__));                                               \
            pt_context_destroy(ctx);                                                                                  \
            return PT_ERR_CUDA;                                                                                       \
        }                                                                                                             \
    } while (0)
    PT_CREATE_CHECK(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
    {
        // a PRIVATE stream-ordered pool that keeps its freed blocks cached (bvh_build.cu: buildAccel makes no driver
        // allocation on a rebuild); the device's default pool — possibly shared with the host application — is untouched
        cudaMemPoolProps props = {};
        props.allocType = cudaMemAllocationTypePinned;
        props.handleTypes = cudaMemHandleTypeNone;
        props.location.type = cudaMemLocationTypeDevice;
        props.location.id = cuda_device;
        PT_CREATE_CHECK(cudaMemPoolCreate(&ctx->memPool, &props));
        uint64_t threshold = UINT64_MAX;
        PT_CREATE_CHECK(cudaMemPoolSetAttribute(ctx->memPool, cudaMemPoolAttrReleaseThreshold, &threshold));
    }
    PT_CREATE_CHECK(cudaEventCreate(&ctx->evStart));
    PT_CREATE_CHECK(cudaEventCreate(&ctx->evStop));
    PT_CREATE_CHECK(cudaMalloc((void **)&ctx->dCounters, sizeof(DeviceCounters)));
    PT_CREATE_CHECK(cudaMemset(ctx->dCounters, 0, sizeof(DeviceCounters)));
    PT_CREATE_CHECK(cudaMalloc((void **)&ctx->dQueueCounts, sizeof(QueueCounts) * PT_MAX_POOLS));
    PT_CREATE_CHECK(cudaMemset(ctx->dQueueCounts, 0, sizeof(QueueCounts) * PT_MAX_POOLS));
    PT_CREATE_CHECK(cudaMallocHost((void **)&ctx->hQueueCounts, sizeof(QueueCounts) * PT_MAX_POOLS));
    PT_CREATE_CHECK(cudaMalloc((void **)&ctx->dNextItem, 4));
    PT_CREATE_CHECK(cudaMallocHost((void **)&ctx->hNextItem, 4));
    PT_CREATE_CHECK(cudaEventCreateWithFlags(&ctx->evRound, cudaEventDisableTiming));
    for (int i = 0; i < PT_MAX_POOLS; i++)
        PT_CREATE_CHECK(cudaStreamCreateWithFlags(&ctx->poolStreams[i], cudaStreamNonBlocking));
    // decode tables: [0..255] UNORM8 -> float, [256..511] sRGB8 -> linear float (same formulas as the oracle)
    float lut[512];
    for (int i = 0; i < 256; i++)
    {
        const double c = i / 255.0;
        lut[i] = (float)i / 255.0f;
        lut[256 + i] = (float)(c <= 0.04045 ? c / 12.92 : std::pow((c + 0.055) / 1.055, 2.4));
    }
    PT_CREATE_CHECK(cudaMalloc((void **)&ctx->dLut, sizeof(lut)));
    PT_CREATE_CHECK(cudaMemcpy(ctx->dLut, lut, sizeof(lut), cudaMemcpyHostToDevice));
#undef PT_CREATE_CHECK
    *out_ctx = ctx;
    return PT_OK;
}

void pt_context_destroy(pt_context *ctx)
{
    if (!ctx)
        return;
    DeviceGuard guard(ctx->device);
    if (ctx->stream)
        cudaStreamSynchronize(ctx->stream);
    freeScene(ctx);
    freeTarget(ctx);
    cudaFree(ctx->dCounters);
    cudaFree(ctx->dQueueCounts);
    cudaFree(ctx->dNextItem);
    if (ctx->hNextItem)
        cudaFreeHost(ctx->hNextItem);
    if (ctx->evRound)
        cudaEventDestroy(ctx->evRound);
    for (int i = 0; i < PT_MAX_POOLS; i++)
        if (ctx->poolStreams[i])
            cudaStreamDestroy(ctx->poolStreams[i]);
    cudaFree(ctx->dLut);
    if (ctx->hQueueCounts)
        cudaFreeHost(ctx->hQueueCounts);
    if (ctx->evStart)
        cudaEventDestroy(ctx->evStart);
    if (ctx->evStop)
        cudaEventDestroy(ctx->evStop);
    if (ctx->stream)
        cudaStreamDestroy(ctx->stream);
    if (ctx->memPool)
        cudaMemPoolDestroy(ctx->memPool);
    delete ctx;
}

const char *pt_last_error(const pt_context *ctx) { return ctx ? ctx->lastError.c_str() : g_createError.c_str(); }

pt_status pt_scene_upload(pt_context *ctx, const pt_scene_desc *scene)
{
    if (!ctx)
        return PT_ERR_INVALID_ARGUMENT;
    ctx->temporalValid = false; // the temporal denoiser's history shows the old scene
    DeviceGuard guard(ctx->device);
    return uploadScene(ctx, scene);
}

pt_status pt_texture_upload(pt_context *ctx, uint32_t slot, const pt_texture_desc *texture)
{
    if (!ctx)
        return PT_ERR_INVALID_ARGUMENT;
    ctx->temporalValid = false; // the temporal denoiser's history shows the old scene
    DeviceGuard guard(ctx->device);
    return uploadTextureSlot(ctx, slot, texture);
}

pt_status pt_render_begin(pt_context *ctx, uint32_t width, uint32_t height)
{
    if (!ctx)
        return PT_ERR_INVALID_ARGUMENT;
    if (width == 0 || height == 0 || (uint64_t)width * height > 0x7fffffffull)
        return fail(ctx, PT_ERR_INVALID_ARGUMENT, "pt_render_begin", "bad extent");
    DeviceGuard guard(ctx->device);
    const size_t n = (size_t)width * height;
    const bool reuse = ctx->accum && ctx->width == width && ctx->height == height;
    if (!reuse)
    {
        PT_CUDA_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
        freeTarget(ctx);
        PathState &ps = ctx->ps;
#define PT_T(expr)                                                                                                    \
    do                                                                                                                \
    {                                                                                                                 \
        const pt_status s__ = (expr);                                                                                 \
        if (s__ != PT_OK)                                                                                             \
        {                                                                                                             \
            freeTarget(ctx);                                                                                          \
            return s__;                                                                                               \
        }                                                                                                             \
    } while (0)
        // slot pool: enough paths in flight to fill the GPU many times over (148 SMs x 2048 threads =
        // 0.3 M resident threads), independent of the image size beyond tiny frames
        size_t slots = ctx->slotPoolSize;
        slots = std::min(slots, std::max<size_t>(n * 4, 4096));
        PT_T(targetAlloc(ctx, &ctx->accum, n));
        PT_T(targetAlloc(ctx, &ctx->pixelList, n));
        PT_T(targetAlloc(ctx, &ps.rec, slots));
        PT_T(targetAlloc(ctx, &ps.contQ[0], slots));
        PT_T(targetAlloc(ctx, &ps.contQ[1], slots));
        PT_T(targetAlloc(ctx, &ps.regenQ[0], slots));
        PT_T(targetAlloc(ctx, &ps.regenQ[1], slots));
        PT_T(targetAlloc(ctx, &ps.hitQ, slots));
        PT_T(targetAlloc(ctx, &ps.hitKey, slots));
        PT_T(targetAlloc(ctx, &ps.hitQSorted, slots));
        PT_T(targetAlloc(ctx, &ps.hitKeySorted, slots));
        {
            const pt_status s__ = allocSortTemp(ctx, slots);
            if (s__ != PT_OK)
            {
                freeTarget(ctx);
                return s__;
            }
        }
        PT_T(targetAlloc(ctx, &ps.shadowQueue, slots));
#undef PT_T
        // the hit sort moves all `slots` (key, value) pairs; the values behind the live entries are never consumed,
        // but they are defined once here so that the sort reads no uninitialised memory (compute-sanitizer initcheck)
        PT_CUDA_CHECK(ctx, cudaMemsetAsync(ps.hitQ, 0, slots * sizeof(*ps.hitQ), ctx->stream));
        PT_CUDA_CHECK(ctx, cudaMemsetAsync(ps.hitQSorted, 0, slots * sizeof(*ps.hitQSorted), ctx->stream));
        ctx->width = width;
        ctx->height = height;
        ctx->slotCapacity = (uint32_t)slots;
    }
    PT_CUDA_CHECK(ctx, cudaMemsetAsync(ctx->accum, 0, n * sizeof(float4), ctx->stream));
    ctx->denoiseValid = false;
    ctx->targetContent = Context::TargetContent::Empty;
    return PT_OK;
}

pt_status pt_render_samples(pt_context *ctx, const pt_render_params *params, uint32_t first_sample, uint32_t sample_count,
                            const pt_tile *tiles, uint32_t tile_count)
{
    if (!ctx)
        return PT_ERR_INVALID_ARGUMENT;
    DeviceGuard guard(ctx->device);
    return renderFrames(ctx, params, first_sample, sample_count, 1, tiles, tile_count);
}

pt_status pt_render_frames(pt_context *ctx, const pt_render_params *params, uint32_t first_sample, uint32_t frame_count,
                           uint32_t samples_per_frame, const pt_tile *tiles, uint32_t tile_count)
{
    if (!ctx)
        return PT_ERR_INVALID_ARGUMENT;
    DeviceGuard guard(ctx->device);
    return renderFrames(ctx, params, first_sample, frame_count, samples_per_frame, tiles, tile_count);
}

pt_status pt_accum_device_ptr(pt_context *ctx, void **out_ptr, size_t *out_pitch, void **out_stream)
{
    if (!ctx)
        return PT_ERR_INVALID_ARGUMENT;
    if (!ctx->accum)
        return fail(ctx, PT_ERR_NO_TARGET, "pt_accum_device_ptr", "pt_render_begin has not been called");
    if (out_ptr)
        *out_ptr = ctx->accum;
    if (out_pitch)
        *out_pitch = (size_t)ctx->width * sizeof(float4);
    if (out_stream)
        *out_stream = ctx->stream;
    return PT_OK;
}

pt_status pt_readback(pt_context *ctx, float *out_rgba, size_t out_bytes)
{
    if (!ctx)
        return PT_ERR_INVALID_ARGUMENT;
    if (!ctx->accum)
        return fail(ctx, PT_ERR_NO_TARGET, "pt_readback", "pt_render_begin has not been called");
    const size_t need = (size_t)ctx->width * ctx->height * sizeof(float4);
    if (!out_rgba || out_bytes < need)
        return fail(ctx, PT_ERR_INVALID_ARGUMENT, "pt_readback", "output buffer too small");
    DeviceGuard guard(ctx->device);
    PT_CUDA_CHECK(ctx, cudaMemcpyAsync(out_rgba, ctx->accum, need, cudaMemcpyDeviceToHost, ctx->stream));
    PT_CUDA_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    return PT_OK;
}

pt_status pt_scene_update(pt_context *ctx, const pt_scene_update_desc *desc)
{
    if (!ctx)
        return PT_ERR_INVALID_ARGUMENT;
    ctx->temporalValid = false; // the temporal denoiser's history shows the old scene
    DeviceGuard guard(ctx->device);
    return updateScene(ctx, desc);
}

pt_status pt_postprocess(pt_context *ctx, const pt_postprocess_params *params, uint32_t total_samples,
                         uint32_t output_format, void *out_pixels, size_t out_bytes)
{
    if (!ctx)
        return PT_ERR_INVALID_ARGUMENT;
    DeviceGuard guard(ctx->device);
    return postProcess(ctx, "pt_postprocess", params, ctx->accum, (float)total_samples, output_format, out_pixels, out_bytes);
}

pt_status pt_denoise(pt_context *ctx, const pt_render_params *params, const pt_denoise_params *denoise_params,
                     uint32_t total_samples, float *out_rgba, size_t out_bytes)
{
    if (!ctx)
        return PT_ERR_INVALID_ARGUMENT;
    DeviceGuard guard(ctx->device);
    return denoise(ctx, "pt_denoise", params, denoise_params, ctx->accum, (float)total_samples, out_rgba, out_bytes);
}

pt_status pt_denoise_guides(pt_context *ctx, float *out_albedo_t, float *out_normal, size_t out_bytes)
{
    if (!ctx)
        return PT_ERR_INVALID_ARGUMENT;
    if (!ctx->accum)
        return fail(ctx, PT_ERR_NO_TARGET, "pt_denoise_guides", "pt_render_begin has not been called");
    if (!ctx->denoiseValid)
        return fail(ctx, PT_ERR_INVALID_ARGUMENT, "pt_denoise_guides", "no pt_denoise since the last pt_render_begin");
    const size_t need = (size_t)ctx->width * ctx->height * sizeof(float4);
    if (out_bytes < need)
        return fail(ctx, PT_ERR_INVALID_ARGUMENT, "pt_denoise_guides", "output buffer too small");
    DeviceGuard guard(ctx->device);
    if (out_albedo_t)
        PT_CUDA_CHECK(ctx, cudaMemcpyAsync(out_albedo_t, ctx->denoiseAlbedoT, need, cudaMemcpyDeviceToHost, ctx->stream));
    if (out_normal)
        PT_CUDA_CHECK(ctx, cudaMemcpyAsync(out_normal, ctx->denoiseNormal, need, cudaMemcpyDeviceToHost, ctx->stream));
    PT_CUDA_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    return PT_OK;
}

pt_status pt_postprocess_denoised(pt_context *ctx, const pt_postprocess_params *params, uint32_t output_format, void *out_pixels,
                                  size_t out_bytes)
{
    if (!ctx)
        return PT_ERR_INVALID_ARGUMENT;
    if (!ctx->accum)
        return fail(ctx, PT_ERR_NO_TARGET, "pt_postprocess_denoised", "pt_render_begin has not been called");
    if (!ctx->denoiseValid)
        return fail(ctx, PT_ERR_INVALID_ARGUMENT, "pt_postprocess_denoised", "no pt_denoise since the last pt_render_begin");
    DeviceGuard guard(ctx->device);
    return postProcess(ctx, "pt_postprocess_denoised", params, ctx->denoised, 1.0f, output_format, out_pixels, out_bytes);
}

pt_status pt_denoise_temporal(pt_context *ctx, const pt_render_params *params, const pt_denoise_params *denoise_params,
                              const pt_temporal_params *temporal, uint32_t total_samples, float *out_rgba, size_t out_bytes)
{
    if (!ctx)
        return PT_ERR_INVALID_ARGUMENT;
    DeviceGuard guard(ctx->device);
    return denoiseTemporal(ctx, params, denoise_params, temporal, total_samples, out_rgba, out_bytes);
}

pt_status pt_denoise_temporal_history(pt_context *ctx, float *out_irradiance_n, float *out_moments, size_t pixels)
{
    if (!ctx)
        return PT_ERR_INVALID_ARGUMENT;
    DeviceGuard guard(ctx->device);
    return temporalHistory(ctx, out_irradiance_n, out_moments, pixels);
}

pt_status pt_render_adaptive(pt_context *ctx, const pt_render_params *params, const pt_adaptive_params *adaptive,
                             pt_adaptive_info *out_info)
{
    if (!ctx)
        return PT_ERR_INVALID_ARGUMENT;
    DeviceGuard guard(ctx->device);
    return renderAdaptive(ctx, params, adaptive, out_info);
}

// the target must hold an adaptive render for the adaptive read functions
static pt_status checkAdaptiveTarget(Context *ctx, const char *what)
{
    if (!ctx->accum)
        return fail(ctx, PT_ERR_NO_TARGET, what, "pt_render_begin has not been called");
    if (ctx->targetContent != Context::TargetContent::Adaptive)
        return fail(ctx, PT_ERR_INVALID_ARGUMENT, what, "no pt_render_adaptive since the last pt_render_begin");
    return PT_OK;
}

pt_status pt_adaptive_readback(pt_context *ctx, uint32_t *out_counts, float *out_mean_m2, size_t pixels)
{
    if (!ctx)
        return PT_ERR_INVALID_ARGUMENT;
    const pt_status s = checkAdaptiveTarget(ctx, "pt_adaptive_readback");
    if (s != PT_OK)
        return s;
    const size_t n = (size_t)ctx->width * ctx->height;
    if (pixels < n)
        return fail(ctx, PT_ERR_INVALID_ARGUMENT, "pt_adaptive_readback", "output buffer too small");
    DeviceGuard guard(ctx->device);
    const AdaptivePixel *px = ctx->adaptivePixels;
    if (out_counts)
        PT_CUDA_CHECK(ctx, cudaMemcpy2DAsync(out_counts, sizeof(uint32_t), &px->count, sizeof(AdaptivePixel), sizeof(uint32_t), n,
                                             cudaMemcpyDeviceToHost, ctx->stream));
    if (out_mean_m2)
        PT_CUDA_CHECK(ctx, cudaMemcpy2DAsync(out_mean_m2, 2 * sizeof(float), &px->mean, sizeof(AdaptivePixel), 2 * sizeof(float), n,
                                             cudaMemcpyDeviceToHost, ctx->stream));
    PT_CUDA_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    return PT_OK;
}

pt_status pt_postprocess_adaptive(pt_context *ctx, const pt_postprocess_params *params, uint32_t output_format, void *out_pixels,
                                  size_t out_bytes)
{
    if (!ctx)
        return PT_ERR_INVALID_ARGUMENT;
    const char *what = "pt_postprocess_adaptive";
    pt_status s = checkPostProcess(ctx, what, params, output_format, out_pixels, out_bytes);
    if (s == PT_OK)
        s = checkAdaptiveTarget(ctx, what);
    if (s != PT_OK)
        return s;
    DeviceGuard guard(ctx->device);
    s = adaptiveMeanImage(ctx, what);
    if (s == PT_OK)
        s = postProcess(ctx, what, params, ctx->adaptiveMean, 1.0f, output_format, out_pixels, out_bytes);
    if (s == PT_OK)
        ctx->stats.kernel_launches++; // k_adaptive_mean
    return s;
}

pt_status pt_denoise_adaptive(pt_context *ctx, const pt_render_params *params, const pt_denoise_params *denoise_params,
                              float *out_rgba, size_t out_bytes)
{
    if (!ctx)
        return PT_ERR_INVALID_ARGUMENT;
    const char *what = "pt_denoise_adaptive";
    pt_status s = checkDenoise(ctx, what, params, denoise_params, 1.0f, out_rgba, out_bytes);
    if (s == PT_OK)
        s = checkAdaptiveTarget(ctx, what);
    if (s != PT_OK)
        return s;
    DeviceGuard guard(ctx->device);
    s = adaptiveMeanImage(ctx, what);
    if (s == PT_OK)
        s = denoise(ctx, what, params, denoise_params, ctx->adaptiveMean, 1.0f, out_rgba, out_bytes);
    if (s == PT_OK)
        ctx->stats.kernel_launches++; // k_adaptive_mean
    return s;
}

pt_status pt_synchronize(pt_context *ctx)
{
    if (!ctx)
        return PT_ERR_INVALID_ARGUMENT;
    DeviceGuard guard(ctx->device);
    PT_CUDA_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    return PT_OK;
}

pt_status pt_first_hit_aov(pt_context *ctx, const pt_render_params *params, uint32_t width, uint32_t height,
                           pt_hit *out_hits)
{
    if (!ctx)
        return PT_ERR_INVALID_ARGUMENT;
    DeviceGuard guard(ctx->device);
    return firstHitAov(ctx, params, width, height, out_hits);
}

pt_status pt_trace_closest(pt_context *ctx, const pt_ray *rays, uint64_t ray_count, pt_hit *out_hits)
{
    if (!ctx)
        return PT_ERR_INVALID_ARGUMENT;
    DeviceGuard guard(ctx->device);
    return traceClosest(ctx, rays, ray_count, out_hits);
}

pt_status pt_trace_occlusion(pt_context *ctx, const pt_ray *rays, uint64_t ray_count, uint8_t *out_occluded)
{
    if (!ctx)
        return PT_ERR_INVALID_ARGUMENT;
    DeviceGuard guard(ctx->device);
    return traceOcclusion(ctx, rays, ray_count, out_occluded);
}

pt_status pt_get_stats(pt_context *ctx, pt_stats *out)
{
    if (!ctx || !out)
        return PT_ERR_INVALID_ARGUMENT;
    DeviceGuard guard(ctx->device);
    DeviceCounters c;
    PT_CUDA_CHECK(ctx, cudaMemcpyAsync(&c, ctx->dCounters, sizeof(c), cudaMemcpyDeviceToHost, ctx->stream));
    PT_CUDA_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    pt_stats s = ctx->stats;
    s.rays_closest = c.raysClosest;
    s.rays_shadow = c.raysShadow;
    s.samples = c.samples;
    s.hits = c.hits;
    s.box_tests_closest = c.boxClosest;
    s.tri_tests_closest = c.triClosest;
    s.alpha_tests_closest = c.alphaClosest;
    s.box_tests_shadow = c.boxShadow;
    s.tri_tests_shadow = c.triShadow;
    s.alpha_tests_shadow = c.alphaShadow;
    s.texel_fetches = c.texels;
    s.restarts = c.restarts;
    for (int i = 0; i < 8; i++)
        s.node_visit_hist[i] = c.visitHist[i];
    s.warp_iterations = c.warpIters;
    s.warp_drain_iterations = c.warpDrainIters;
    s.max_warp_drain_iterations = c.maxWarpDrainIters;
    s.triangle_count = ctx->scene.triCount ? ctx->triangleCount : 0;
    s.bvh_reference_count = ctx->scene.triCount;
    s.bvh_node_count = ctx->nodeCount;
    s.bvh_bytes = ctx->bvhBytes;
    s.bvh_max_depth = ctx->bvhMaxDepth;
    s.bvh_build_ms = ctx->bvhBuildMs;
    s.scene_upload_ms = ctx->sceneUploadMs;
    *out = s;
    return PT_OK;
}

pt_status pt_set_traversal_stats(pt_context *ctx, int32_t enable)
{
    if (!ctx)
        return PT_ERR_INVALID_ARGUMENT;
    ctx->collectTraversalStats = enable != 0;
    return PT_OK;
}

pt_status pt_set_kernel_timing(pt_context *ctx, int32_t enable)
{
    if (!ctx)
        return PT_ERR_INVALID_ARGUMENT;
    ctx->kernelTiming = enable != 0;
    return PT_OK;
}

pt_status pt_set_tuning(pt_context *ctx, const char *key, uint64_t value)
{
    if (!ctx || !key)
        return PT_ERR_INVALID_ARGUMENT;
    const std::string k(key);
    if (k == "pools")
        ctx->poolCount = (uint32_t)std::min<uint64_t>(PT_MAX_POOLS, std::max<uint64_t>(1, value));
    else if (k == "slots")
    {
        ctx->slotPoolSize = std::max<uint64_t>(1024, value);
        if (ctx->accum)
        {
            // re-create the path state with the new pool size
            const uint32_t w = ctx->width, h = ctx->height;
            DeviceGuard guard(ctx->device);
            PT_CUDA_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
            freeTarget(ctx);
            return pt_render_begin(ctx, w, h);
        }
    }
    else if (k == "sort_hits")
        ctx->sortHits = value != 0;
    else if (k == "bvh_builder") // takes effect at the next pt_scene_upload
        ctx->bvhBuilder = value != 0;
    else if (k == "ploc_radius")
        ctx->plocRadius = (uint32_t)std::max<uint64_t>(1, value);
    else if (k == "split_threshold_x100") // reference splitting; takes effect at the next upload / update
        ctx->splitThreshold = (float)value / 100.0f;
    else if (k == "max_texture_size") // TextureUploader::MaxTextureDataSize (4096); takes effect at the next upload
        ctx->maxTextureSize = (uint32_t)std::min<uint64_t>(32768, std::max<uint64_t>(1, value));
    else if (k == "texture_budget_mb") // Config::MaxTextureMemoryBudget*; 0 = ForceFullTextureSize (default)
        ctx->textureBudgetBytes = value << 20;
    else if (k == "sbuf_mb")
        ctx->sbufBudgetBytes = std::max<uint64_t>(1, value) << 20;
    else
        return fail(ctx, PT_ERR_INVALID_ARGUMENT, "pt_set_tuning", "unknown key");
    return PT_OK;
}

pt_status pt_set_sampler(pt_context *ctx, uint32_t max_anisotropy)
{
    if (!ctx)
        return PT_ERR_INVALID_ARGUMENT;
    if (max_anisotropy < 1 || max_anisotropy > 16)
        return fail(ctx, PT_ERR_INVALID_ARGUMENT, "pt_set_sampler", "max_anisotropy must be in 1..16");
    ctx->maxAnisotropy = max_anisotropy;
    ctx->scene.maxAnisotropy = max_anisotropy; // the scene struct travels to every kernel by value
    ctx->emittersValid = false;                // emitter weights are textureGrad fetches
    return PT_OK;
}

pt_status pt_set_light_sampling(pt_context *ctx, uint32_t mode)
{
    if (!ctx)
        return PT_ERR_INVALID_ARGUMENT;
    if (mode != PT_LIGHT_SAMPLING_REFERENCE && mode != PT_LIGHT_SAMPLING_EMISSIVE_MIS)
        return fail(ctx, PT_ERR_INVALID_ARGUMENT, "pt_set_light_sampling", "unknown light-sampling mode");
    ctx->lightSampling = mode;
    return PT_OK;
}

pt_status pt_emitter_table(pt_context *ctx, uint32_t *out_count, uint32_t *flat_ids, uint32_t *weights,
                           uint32_t *alias_threshold, uint32_t *alias_index, uint32_t capacity)
{
    if (!ctx || !out_count)
        return PT_ERR_INVALID_ARGUMENT;
    if (!ctx->hasScene)
        return fail(ctx, PT_ERR_NO_SCENE, "pt_emitter_table", "no scene uploaded");
    DeviceGuard guard(ctx->device);
    if (!ctx->emittersValid)
    {
        const pt_status st = buildEmitters(ctx);
        if (st != PT_OK)
            return st;
    }
    const uint32_t n = ctx->emitters.count;
    *out_count = n;
    if ((flat_ids || weights || alias_threshold || alias_index) && capacity < n)
        return fail(ctx, PT_ERR_INVALID_ARGUMENT, "pt_emitter_table", "capacity is below the emitter count");
    for (uint32_t k = 0; k < n; k++)
    {
        if (flat_ids)
            flat_ids[k] = ctx->emitterIds[k];
        if (weights)
            weights[k] = ctx->emitterWeights[k];
        if (alias_threshold)
            alias_threshold[k] = ctx->emitterAlias[k].x;
        if (alias_index)
            alias_index[k] = ctx->emitterAlias[k].y;
    }
    return PT_OK;
}

pt_status pt_debug_render(pt_context *ctx, const pt_render_params *params, const pt_debug_params *debug, uint32_t width,
                          uint32_t height, float *out_rgba)
{
    if (!ctx)
        return PT_ERR_INVALID_ARGUMENT;
    DeviceGuard guard(ctx->device);
    return debugRender(ctx, params, debug, width, height, out_rgba);
}

pt_status pt_test_texture(pt_context *ctx, uint32_t slot, const float *in6, float *out4, uint32_t count, int32_t use_grad)
{
    if (!ctx)
        return PT_ERR_INVALID_ARGUMENT;
    DeviceGuard guard(ctx->device);
    return testTexture(ctx, slot, in6, out4, count, use_grad);
}

pt_status pt_test_trace(pt_context *ctx, const pt_ray *rays, uint64_t ray_count, uint32_t flags, uint32_t blocks, pt_hit *out_hits,
                        float *out_decals, uint64_t *out_tail)
{
    if (!ctx)
        return PT_ERR_INVALID_ARGUMENT;
    DeviceGuard guard(ctx->device);
    return testTrace(ctx, rays, ray_count, flags, blocks, out_hits, out_decals, out_tail);
}

uint32_t pt_test_input_stride(uint32_t mode) { return testInputStride(mode); }
uint32_t pt_test_output_stride(uint32_t mode) { return testOutputStride(mode); }

pt_status pt_test_shading(pt_context *ctx, uint32_t mode, const float *input, float *output, uint32_t count)
{
    if (!ctx)
        return PT_ERR_INVALID_ARGUMENT;
    DeviceGuard guard(ctx->device);
    return testShading(ctx, mode, input, output, count);
}

} // extern "C"
