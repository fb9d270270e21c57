// postprocess.cu — post-processing and output conversion of the accumulated image (SURVEY §8f rank 2).
//
// Replaces Renderer::RecordPostProcessCommands (PT/Renderer/Renderer.cpp:928-1060), the offline
// branch Renderer::RecordSaveOutputCommands (:1205-1250) and OutputSaver's final blit
// (PT/Renderer/OutputSaver.cpp:113-140).  One kernel per reference dispatch:
//   k_post_prefilter   postprocess.comp:16-40      sum / samples * exposure, NaN / Inf markers, bloom prefilter
//   k_bloom_down       bloomDownsample.comp:18-58  13-tap downsample, level i -> i + 1
//   k_bloom_up         bloomUpsample.comp:18-52    3x3 tent upsample, level i -> i - 1 (added)
//   k_post_output      composition.comp:15-25 + toneMapping.comp:13-24 + the blit to the output format
// Every image of the chain is RGBA16F in the reference; here each is an array of __half2 pairs
// (rg, b1) and every store rounds to half like imageStore does.  All of it is HBM streaming:
// 16 B read + 16 B written per pixel for the first pass, 8-byte texels afterwards.
#include "core_internal.h"

#include <cuda_fp16.h>

#include <algorithm>

namespace pt
{

namespace
{

struct HalfLevel
{
    uint2 *px; // one RGBA16F texel: x = (r, g), y = (b, a) as __half2 bits
    uint32_t w, h;
};

__device__ __forceinline__ float roundHalf(float f) { return __half2float(__float2half_rn(f)); }

__device__ __forceinline__ uint2 packTexel(float r, float g, float b)
{
    const __half2 rg = __floats2half2_rn(r, g), ba = __floats2half2_rn(b, 1.0f);
    uint2 t;
    t.x = *reinterpret_cast<const uint32_t *>(&rg);
    t.y = *reinterpret_cast<const uint32_t *>(&ba);
    return t;
}

__device__ __forceinline__ float3 unpackTexel(uint2 t)
{
    const float2 rg = __half22float2(*reinterpret_cast<const __half2 *>(&t.x));
    const float2 ba = __half22float2(*reinterpret_cast<const __half2 *>(&t.y));
    return make_float3(rg.x, rg.y, ba.x);
}

__device__ __forceinline__ float3 add3(float3 a, float3 b) { return make_float3(a.x + b.x, a.y + b.y, a.z + b.z); }
__device__ __forceinline__ float3 mul3(float3 a, float s) { return make_float3(a.x * s, a.y * s, a.z * s); }

// texture(sampler2D, uv) with Renderer.cpp:114-119's bloom sampler: linear, clamp to edge
__device__ __forceinline__ float3 sampleLevel(const HalfLevel &l, float u, float v)
{
    const float x = u * (float)l.w - 0.5f, y = v * (float)l.h - 0.5f;
    const float fx0 = floorf(x), fy0 = floorf(y);
    const float fx = x - fx0, fy = y - fy0;
    const int x0 = min(max((int)fx0, 0), (int)l.w - 1), x1 = min(max((int)fx0 + 1, 0), (int)l.w - 1);
    const int y0 = min(max((int)fy0, 0), (int)l.h - 1), y1 = min(max((int)fy0 + 1, 0), (int)l.h - 1);
    const float3 t00 = unpackTexel(__ldg(l.px + (size_t)y0 * l.w + x0)), t10 = unpackTexel(__ldg(l.px + (size_t)y0 * l.w + x1));
    const float3 t01 = unpackTexel(__ldg(l.px + (size_t)y1 * l.w + x0)), t11 = unpackTexel(__ldg(l.px + (size_t)y1 * l.w + x1));
    const float3 top = add3(mul3(t00, 1.0f - fx), mul3(t10, fx));
    const float3 bot = add3(mul3(t01, 1.0f - fx), mul3(t11, fx));
    return add3(mul3(top, 1.0f - fy), mul3(bot, fy));
}

__global__ void __launch_bounds__(256) k_post_prefilter(const float4 *__restrict__ accum, uint32_t n, float totalSamples,
                                                        float exposure, float threshold, uint2 *__restrict__ color,
                                                        uint2 *__restrict__ bloom)
{
    const uint32_t stride = gridDim.x * blockDim.x;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
    {
        const float4 a = __ldg(accum + i);
        float r = a.x / totalSamples * exposure, g = a.y / totalSamples * exposure, b = a.z / totalSamples * exposure;
        if (isnan(r) || isnan(g) || isnan(b))
            r = 5000.0f, g = 0.0f, b = 0.0f;
        if (isinf(r) || isinf(g) || isinf(b))
            r = 0.0f, g = 5000.0f, b = 0.0f;
        const float knee = 0.5f;
        const float br = fmaxf(r, fmaxf(g, b));
        const float cx = threshold - knee, cy = knee * 2.0f, cz = 0.25f / knee;
        float rq = fminf(fmaxf(br - cx, 0.0f), cy);
        rq = cz * rq * rq;
        const float w = fmaxf(rq, br - threshold) / fmaxf(br, 0.0001f);
        color[i] = packTexel(r, g, b);
        bloom[i] = packTexel(r * w, g * w, b * w);
    }
}

__global__ void __launch_bounds__(256) k_bloom_down(HalfLevel src, HalfLevel dst)
{
    const uint32_t x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= dst.w || y >= dst.h)
        return;
    const float tx = 1.0f / (float)src.w, ty = 1.0f / (float)src.h;
    const float u = ((float)x + 0.5f) / (float)dst.w, v = ((float)y + 0.5f) / (float)dst.h;
    auto tap = [&](float ox, float oy) { return sampleLevel(src, u + ox * tx, v + oy * ty); };
    const float3 a = tap(-2, 2), b = tap(0, 2), c = tap(2, 2);
    const float3 d = tap(-2, 0), e = tap(0, 0), f = tap(2, 0);
    const float3 g = tap(-2, -2), h = tap(0, -2), i = tap(2, -2);
    const float3 j = tap(-1, 1), k = tap(1, 1), l = tap(-1, -1), m = tap(1, -1);
    float3 down = mul3(e, 0.125f);
    down = add3(down, mul3(add3(add3(add3(a, c), g), i), 0.03125f));
    down = add3(down, mul3(add3(add3(add3(b, d), f), h), 0.0625f));
    down = add3(down, mul3(add3(add3(add3(j, k), l), m), 0.125f));
    dst.px[(size_t)y * dst.w + x] = packTexel(down.x, down.y, down.z);
}

__global__ void __launch_bounds__(256) k_bloom_up(HalfLevel src, HalfLevel dst)
{
    const uint32_t x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= dst.w || y >= dst.h)
        return;
    const float tx = 1.0f / (float)src.w, ty = 1.0f / (float)src.h;
    const float u = ((float)x + 0.5f) / (float)dst.w, v = ((float)y + 0.5f) / (float)dst.h;
    auto tap = [&](float ox, float oy) { return sampleLevel(src, u + ox * tx, v + oy * ty); };
    const float3 a = tap(-1, 1), b = tap(0, 1), c = tap(1, 1);
    const float3 d = tap(-1, 0), e = tap(0, 0), f = tap(1, 0);
    const float3 g = tap(-1, -1), h = tap(0, -1), i = tap(1, -1);
    float3 up = mul3(e, 4.0f);
    up = add3(up, mul3(add3(add3(add3(b, d), f), h), 2.0f));
    up = add3(up, add3(add3(add3(a, c), g), i));
    up = mul3(up, 1.0f / 16.0f);
    uint2 *o = dst.px + (size_t)y * dst.w + x;
    const float3 sum = add3(unpackTexel(*o), up);
    *o = packTexel(sum.x, sum.y, sum.z);
}

// VK_FORMAT_R8G8B8A8_SRGB store of a linear value
__device__ __forceinline__ uint32_t encodeSrgb8(float c)
{
    if (!(c > 0.0f))
        return 0u;
    if (c >= 1.0f)
        return 255u;
    const double l = c;
    const double e = l <= 0.0031308 ? 12.92 * l : 1.055 * pow(l, 1.0 / 2.4) - 0.055;
    return (uint32_t)__double2int_rn(e * 255.0);
}

__global__ void __launch_bounds__(256) k_post_output(const uint2 *__restrict__ color, const uint2 *__restrict__ bloom, uint32_t n,
                                                     float bloomIntensity, uint32_t toneMapping, uint32_t outputFormat,
                                                     void *__restrict__ out)
{
    const uint32_t stride = gridDim.x * blockDim.x;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
    {
        const float3 c0 = unpackTexel(__ldg(color + i)), bl = unpackTexel(__ldg(bloom + i));
        const float k = bloomIntensity * 0.1f;
        float3 c = make_float3(roundHalf(k * bl.x + 1.0f * c0.x), roundHalf(k * bl.y + 1.0f * c0.y), roundHalf(k * bl.z + 1.0f * c0.z));
        if (toneMapping == PT_TONE_MAPPING_SDR)
        {
            c.x = roundHalf((float)(1.0 - exp(-(double)c.x)));
            c.y = roundHalf((float)(1.0 - exp(-(double)c.y)));
            c.z = roundHalf((float)(1.0 - exp(-(double)c.z)));
        }
        if (outputFormat == PT_OUTPUT_RGBA8_SRGB)
            reinterpret_cast<uint32_t *>(out)[i] = encodeSrgb8(c.x) | (encodeSrgb8(c.y) << 8) | (encodeSrgb8(c.z) << 16) | 0xff000000u;
        else
            reinterpret_cast<float4 *>(out)[i] = make_float4(c.x, c.y, c.z, 1.0f);
    }
}

} // namespace

pt_status checkPostProcess(Context *ctx, const char *what, const pt_postprocess_params *p, uint32_t outputFormat, const void *out,
                           size_t outBytes)
{
    if (!p || !out)
        return fail(ctx, PT_ERR_INVALID_ARGUMENT, what, "NULL argument");
    if (!ctx->accum)
        return fail(ctx, PT_ERR_NO_TARGET, what, "pt_render_begin has not been called");
    if (outputFormat != PT_OUTPUT_RGBA8_SRGB && outputFormat != PT_OUTPUT_RGBAF32)
        return fail(ctx, PT_ERR_INVALID_ARGUMENT, what, "unknown output format");
    if (p->tone_mapping > PT_TONE_MAPPING_HDR)
        return fail(ctx, PT_ERR_INVALID_ARGUMENT, what, "unknown tone-mapping mode");
    const size_t need = (size_t)ctx->width * ctx->height * (outputFormat == PT_OUTPUT_RGBA8_SRGB ? 4 : 16);
    if (outBytes < need)
        return fail(ctx, PT_ERR_INVALID_ARGUMENT, what, "output buffer too small");
    return PT_OK;
}

pt_status postProcess(Context *ctx, const char *what, const pt_postprocess_params *p, const float4 *src, float divisor,
                      uint32_t outputFormat, void *out, size_t outBytes)
{
    const pt_status checked = checkPostProcess(ctx, what, p, outputFormat, out, outBytes);
    if (checked != PT_OK)
        return checked;
    const uint32_t W = ctx->width, H = ctx->height;
    const size_t n = (size_t)W * H, need = n * (outputFormat == PT_OUTPUT_RGBA8_SRGB ? 4 : 16);

    // floor(log2(max(w, h))) + 1 levels (PT/Renderer/Image.cpp:14-17)
    uint32_t levels = 1;
    for (uint32_t m = std::max(W, H); m > 1; m >>= 1)
        levels++;
    // Renderer.cpp:955-956 computes min(levels - 3, 12) in unsigned arithmetic and would index
    // non-existent levels for frames smaller than 8 pixels; such frames get no bloom passes here
    const uint32_t maxMip = levels > 3 ? std::min(levels - 3, 12u) : 1u;
    std::vector<HalfLevel> bloom(maxMip);
    size_t texels = 0;
    for (uint32_t l = 0; l < maxMip; l++)
    {
        bloom[l].w = std::max(1u, W >> l);
        bloom[l].h = std::max(1u, H >> l);
        texels += (size_t)bloom[l].w * bloom[l].h;
    }
    uint2 *mem = nullptr;
    void *dOut = nullptr;
    // stream-ordered pool (see bvh_build.cu): repeated calls at one extent make no driver allocation
    cudaStream_t st = ctx->stream;
    PT_CUDA_CHECK(ctx, poolAlloc(ctx, (void **)&mem, (n + texels) * sizeof(uint2), st));
    cudaError_t err = poolAlloc(ctx, &dOut, need, st);
    if (err != cudaSuccess)
    {
        cudaFreeAsync(mem, st);
        PT_CUDA_CHECK(ctx, err);
    }
    uint2 *color = mem, *cursor = mem + n;
    for (uint32_t l = 0; l < maxMip; l++)
    {
        bloom[l].px = cursor;
        cursor += (size_t)bloom[l].w * bloom[l].h;
    }
    const uint32_t wide = (uint32_t)std::min<size_t>((n + 255) / 256, (size_t)ctx->smCount * 8);
    k_post_prefilter<<<wide, 256, 0, st>>>(src, (uint32_t)n, divisor, p->exposure, p->bloom_threshold, color,
                                           bloom[0].px);
    const dim3 block(32, 8);
    for (uint32_t i = 0; i + 1 < maxMip; i++)
    {
        const dim3 grid((bloom[i + 1].w + 31) / 32, (bloom[i + 1].h + 7) / 8);
        k_bloom_down<<<grid, block, 0, st>>>(bloom[i], bloom[i + 1]);
    }
    for (uint32_t i = maxMip - 1; i > 0; i--)
    {
        const dim3 grid((bloom[i - 1].w + 31) / 32, (bloom[i - 1].h + 7) / 8);
        k_bloom_up<<<grid, block, 0, st>>>(bloom[i], bloom[i - 1]);
    }
    k_post_output<<<wide, 256, 0, st>>>(color, bloom[0].px, (uint32_t)n, p->bloom_intensity, p->tone_mapping, outputFormat, dOut);
    err = cudaGetLastError();
    if (err == cudaSuccess)
        err = cudaMemcpyAsync(out, dOut, need, cudaMemcpyDeviceToHost, st);
    if (err == cudaSuccess)
        err = cudaStreamSynchronize(st);
    cudaFreeAsync(mem, st);
    cudaFreeAsync(dOut, st);
    PT_CUDA_CHECK(ctx, err);
    ctx->stats.kernel_launches = 2 + 2 * (uint64_t)(maxMip - 1);
    return PT_OK;
}

} // namespace pt
