// adaptive.cu — adaptive sampling: converged 8x4 pixel blocks stop early (DESIGN.md §3i).
//
// Per pixel the target keeps (count, mean, M2), Welford statistics of the luminance of its samples, which
// k_resolve<true> (wavefront.cu) updates in sample order while it accumulates.  A pass:
//   k_adaptive_blocks   the stop rule per 8x4 block; the smallest count n among the active blocks
//   k_adaptive_select   per block its pixel count if it is active at count n, and the next larger count among the active
//   + exclusive scan    blocks; a device-wide scan of those counts places each block's pixels in ascending block order
//   k_adaptive_scatter  the pass's pixel list, with the full-frame list's in-block order
//   rounds              samples [n, n + k) of those pixels through the unchanged path kernels
// k_adaptive_mean writes accum / count for the post-process chain and the denoiser.
// tests/adaptive_ref.py is the numpy reference of the statistics, the stop rule and the pass schedule.
#include "core_internal.h"

#include <cub/device/device_scan.cuh>

#include <algorithm>
#include <cmath>

namespace pt
{

namespace
{

constexpr uint32_t kNone = 0xffffffffu; // an inactive block's word; "no count" in the summary
constexpr uint32_t kBlockW = 8, kBlockH = 4;
constexpr uint64_t kDefaultMinPassItems = 1ull << 21;

// relative standard error of the mean <= t against the relMSE denominator mean^2 + 0.01, without a division or a root
__device__ __forceinline__ bool converged(const AdaptivePixel &p, float t)
{
    return p.m2 <= t * t * (p.mean * p.mean + 0.01f) * (float)p.count * (float)(p.count - 1);
}

// one thread per block: its word is its count if it is active, kNone otherwise
__global__ void __launch_bounds__(256) k_adaptive_blocks(const AdaptivePixel *__restrict__ px, uint32_t W, uint32_t H, uint32_t minSamples,
                                                         uint32_t maxSamples, float t, uint32_t *__restrict__ blocks,
                                                         AdaptiveSummary *__restrict__ sum)
{
    const uint32_t bw = (W + kBlockW - 1) / kBlockW, nb = bw * ((H + kBlockH - 1) / kBlockH);
    const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t activeCount = kNone, minCount = kNone, maxCount = 0, unconverged = 0;
    if (b < nb)
    {
        const uint32_t by = b / bw, bx = b - by * bw;
        const uint32_t x0 = bx * kBlockW, y0 = by * kBlockH, x1 = min(x0 + kBlockW, W), y1 = min(y0 + kBlockH, H);
        const uint32_t count = px[(size_t)y0 * W + x0].count; // the pixels of a block share their count
        uint32_t bad = 0;
        for (uint32_t y = y0; y < y1; y++)
        {
            const AdaptivePixel *row = px + (size_t)y * W;
#pragma unroll
            for (uint32_t dx = 0; dx < kBlockW; dx++)
                if (x0 + dx < x1)
                    bad += converged(row[x0 + dx], t) ? 0u : 1u;
        }
        const bool active = count < minSamples || (count < maxSamples && bad > 0);
        blocks[b] = active ? count : kNone;
        activeCount = active ? count : kNone;
        minCount = maxCount = count;
        unconverged = count >= maxSamples ? bad : 0u;
    }
    activeCount = __reduce_min_sync(0xffffffffu, activeCount);
    minCount = __reduce_min_sync(0xffffffffu, minCount);
    maxCount = __reduce_max_sync(0xffffffffu, maxCount);
    unconverged = __reduce_add_sync(0xffffffffu, unconverged);
    if ((threadIdx.x & 31u) == 0)
    {
        if (activeCount != kNone)
            atomicMin(&sum->n, activeCount);
        if (minCount != kNone)
        {
            atomicMin(&sum->minCount, minCount);
            atomicMax(&sum->maxCount, maxCount);
        }
        if (unconverged)
            atomicAdd(&sum->unconverged, unconverged);
    }
}

// Per block: its pixel count if it is active at count n, else 0 (the input of the exclusive scan that places each block's
// pixels in ascending block order); the next larger count among the active blocks
__global__ void __launch_bounds__(256) k_adaptive_select(const uint32_t *__restrict__ blocks, uint32_t W, uint32_t H,
                                                         uint32_t *__restrict__ counts, AdaptiveSummary *__restrict__ sum)
{
    const uint32_t bw = (W + kBlockW - 1) / kBlockW, nb = bw * ((H + kBlockH - 1) / kBlockH);
    const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t n = sum->n;
    uint32_t next = kNone;
    if (b < nb)
    {
        const uint32_t word = blocks[b], by = b / bw, bx = b - by * bw;
        const uint32_t pixels = (min(bx * kBlockW + kBlockW, W) - bx * kBlockW) * (min(by * kBlockH + kBlockH, H) - by * kBlockH);
        counts[b] = n != kNone && word == n ? pixels : 0u;
        if (word != kNone && word > n)
            next = word;
    }
    next = __reduce_min_sync(0xffffffffu, next);
    if ((threadIdx.x & 31u) == 0 && next != kNone)
        atomicMin(&sum->next, next);
}

// One thread per (block, pixel of the block): a selected block's pixels go to offsets[b] + their in-block raster index, the
// order of the full-frame list, so a warp writes one block's pixels to consecutive words
__global__ void __launch_bounds__(256) k_adaptive_scatter(const uint32_t *__restrict__ counts, const uint32_t *__restrict__ offsets,
                                                          uint32_t W, uint32_t H, uint32_t *__restrict__ pixelList,
                                                          AdaptiveSummary *__restrict__ sum)
{
    const uint32_t bw = (W + kBlockW - 1) / kBlockW, nb = bw * ((H + kBlockH - 1) / kBlockH);
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x, b = t / (kBlockW * kBlockH), l = t % (kBlockW * kBlockH);
    if (b >= nb)
        return;
    if (b + 1 == nb && l == 0)
        sum->pixels = offsets[b] + counts[b];
    if (counts[b] == 0)
        return;
    const uint32_t by = b / bw, bx = b - by * bw, x0 = bx * kBlockW, y0 = by * kBlockH;
    const uint32_t width = min(x0 + kBlockW, W) - x0, height = min(y0 + kBlockH, H) - y0;
    const uint32_t lx = l % kBlockW, ly = l / kBlockW;
    if (lx < width && ly < height)
        pixelList[offsets[b] + ly * width + lx] = (y0 + ly) * W + x0 + lx;
}

__global__ void __launch_bounds__(256) k_adaptive_mean(const float4 *__restrict__ accum, const AdaptivePixel *__restrict__ px, uint32_t n,
                                                       float4 *__restrict__ out)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n)
        return;
    const float4 a = accum[i];
    const float c = (float)px[i].count;
    out[i] = make_float4(a.x / c, a.y / c, a.z / c, 1.0f);
}

} // namespace

pt_status renderAdaptive(Context *ctx, const pt_render_params *params, const pt_adaptive_params *ap, pt_adaptive_info *info)
{
    const char *what = "pt_render_adaptive";
    if (!params || !ap)
        return fail(ctx, PT_ERR_INVALID_ARGUMENT, what, "NULL argument");
    if (!ctx->hasScene)
        return fail(ctx, PT_ERR_NO_SCENE, what, "no scene uploaded");
    if (!ctx->accum)
        return fail(ctx, PT_ERR_NO_TARGET, what, "pt_render_begin has not been called");
    if (params->bounce_count == 0 || params->bounce_count > 255)
        return fail(ctx, PT_ERR_INVALID_ARGUMENT, what, "bounce_count must be in 1..255");
    if (ap->min_samples < 2)
        return fail(ctx, PT_ERR_INVALID_ARGUMENT, what, "min_samples must be at least 2");
    if (ap->max_samples < ap->min_samples)
        return fail(ctx, PT_ERR_INVALID_ARGUMENT, what, "max_samples must be at least min_samples");
    if (ap->batch == 0)
        return fail(ctx, PT_ERR_INVALID_ARGUMENT, what, "batch must be at least 1");
    if (!std::isfinite(ap->threshold) || ap->threshold < 0.0f)
        return fail(ctx, PT_ERR_INVALID_ARGUMENT, what, "threshold must be finite and non-negative");
    if (ctx->targetContent == Context::TargetContent::Uniform)
        return fail(ctx, PT_ERR_INVALID_ARGUMENT, what,
                    "the target holds a uniform render (unknown per-pixel counts); call pt_render_begin first");
    if (ctx->lightSampling == PT_LIGHT_SAMPLING_EMISSIVE_MIS && !ctx->emittersValid)
    {
        const pt_status st = buildEmitters(ctx);
        if (st != PT_OK)
            return st;
    }

    const uint32_t W = ctx->width, H = ctx->height;
    const size_t n = (size_t)W * H;
    const uint32_t blockCount = ((W + kBlockW - 1) / kBlockW) * ((H + kBlockH - 1) / kBlockH);
    cudaStream_t st = ctx->stream;
    if (!ctx->adaptivePixels)
    {
        // belongs to the target: freeTarget releases it with the accumulation
        size_t scanBytes = 0;
        PT_CUDA_CHECK(ctx, cub::DeviceScan::ExclusiveSum(nullptr, scanBytes, (const uint32_t *)nullptr, (uint32_t *)nullptr,
                                                         (int)blockCount, st));
        scanBytes = (scanBytes + 255) & ~(size_t)255;
        char *mem = nullptr;
        const size_t blockBytes = ((size_t)blockCount * 4 + 255) & ~(size_t)255;
        PT_CUDA_CHECK(ctx, cudaMalloc((void **)&mem, n * sizeof(AdaptivePixel) + 3 * blockBytes + scanBytes + sizeof(AdaptiveSummary)));
        ctx->targetAllocs.push_back(mem);
        char *cursor = mem;
        ctx->adaptivePixels = reinterpret_cast<AdaptivePixel *>(cursor);
        cursor += n * sizeof(AdaptivePixel);
        ctx->adaptiveBlocks = reinterpret_cast<uint32_t *>(cursor);
        ctx->adaptiveCounts = reinterpret_cast<uint32_t *>(cursor + blockBytes);
        ctx->adaptiveOffsets = reinterpret_cast<uint32_t *>(cursor + 2 * blockBytes);
        cursor += 3 * blockBytes;
        ctx->adaptiveScanTemp = cursor;
        ctx->adaptiveScanBytes = scanBytes;
        ctx->adaptiveSummary = reinterpret_cast<AdaptiveSummary *>(cursor + scanBytes);
    }
    if (ctx->targetContent != Context::TargetContent::Adaptive)
        PT_CUDA_CHECK(ctx, cudaMemsetAsync(ctx->adaptivePixels, 0, n * sizeof(AdaptivePixel), st));
    ctx->targetContent = Context::TargetContent::Adaptive;
    ctx->pixelListValid = false; // ctx->pixelList now holds the passes' lists, not a tile set's

    pt_status status = resetRenderStats(ctx);
    if (status != PT_OK)
        return status;
    const uint64_t minPassItems = ap->min_pass_items ? ap->min_pass_items : kDefaultMinPassItems;
    uint32_t passes = 0;
    uint64_t samples = 0;
    AdaptiveSummary hs;
    for (;;)
    {
        // evaluate every block with this call's parameters
        const AdaptiveSummary init = { kNone, kNone, 0, kNone, 0, 0, { 0, 0 } };
        PT_CUDA_CHECK(ctx, cudaMemcpyAsync(ctx->adaptiveSummary, &init, sizeof(init), cudaMemcpyHostToDevice, st));
        k_adaptive_blocks<<<(blockCount + 255) / 256, 256, 0, st>>>(ctx->adaptivePixels, W, H, ap->min_samples, ap->max_samples,
                                                                    ap->threshold, ctx->adaptiveBlocks, ctx->adaptiveSummary);
        k_adaptive_select<<<(blockCount + 255) / 256, 256, 0, st>>>(ctx->adaptiveBlocks, W, H, ctx->adaptiveCounts, ctx->adaptiveSummary);
        size_t scanBytes = ctx->adaptiveScanBytes;
        PT_CUDA_CHECK(ctx, cub::DeviceScan::ExclusiveSum(ctx->adaptiveScanTemp, scanBytes, ctx->adaptiveCounts, ctx->adaptiveOffsets,
                                                         (int)blockCount, st));
        k_adaptive_scatter<<<(uint32_t)(((size_t)blockCount * kBlockW * kBlockH + 255) / 256), 256, 0, st>>>(
            ctx->adaptiveCounts, ctx->adaptiveOffsets, W, H, ctx->pixelList, ctx->adaptiveSummary);
        ctx->stats.kernel_launches += 4; // blocks, select, scan, scatter
        PT_CUDA_CHECK(ctx, cudaMemcpyAsync(&hs, ctx->adaptiveSummary, sizeof(hs), cudaMemcpyDeviceToHost, st));
        PT_CUDA_CHECK(ctx, cudaStreamSynchronize(st));
        if (hs.n == kNone)
            break;
        // samples [n, n + k): up to the next count level, the cap, and at least a batch, min_samples and min_pass_items
        const uint64_t level = hs.n;
        const uint64_t want = std::max({ level + ap->batch, (uint64_t)ap->min_samples, level + (minPassItems + hs.pixels - 1) / hs.pixels });
        const uint64_t to = std::min({ (uint64_t)ap->max_samples, (uint64_t)hs.next, want });
        const uint32_t k = (uint32_t)(to - level);
        ctx->pixelCount = hs.pixels;
        uint32_t roundMax = 0;
        status = sizeSampleBuffer(ctx, k, roundMax);
        if (status == PT_OK)
            status = renderRounds(ctx, params, hs.n, k, 1, roundMax, true);
        if (status != PT_OK)
            return status;
        passes++;
        samples += (uint64_t)hs.pixels * k;
    }
    status = finishRender(ctx, what);
    if (status != PT_OK)
        return status;
    if (info)
    {
        info->passes = passes;
        info->min_count = hs.minCount;
        info->max_count = hs.maxCount;
        info->unconverged_pixels = hs.unconverged;
        info->samples = samples;
    }
    return PT_OK;
}

pt_status adaptiveMeanImage(Context *ctx, const char *what)
{
    const size_t n = (size_t)ctx->width * ctx->height;
    if (!ctx->adaptiveMean)
    {
        // belongs to the target: freeTarget releases it with the accumulation
        PT_CUDA_CHECK(ctx, cudaMalloc((void **)&ctx->adaptiveMean, n * sizeof(float4)));
        ctx->targetAllocs.push_back(ctx->adaptiveMean);
    }
    k_adaptive_mean<<<(uint32_t)((n + 255) / 256), 256, 0, ctx->stream>>>(ctx->accum, ctx->adaptivePixels, (uint32_t)n, ctx->adaptiveMean);
    const cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess)
        return fail(ctx, PT_ERR_CUDA, what, cudaGetErrorString(err));
    return PT_OK;
}

} // namespace pt
