// denoise.cu — edge-avoiding a-trous denoiser of the accumulated image (DESIGN §3h).
//
// SVGF's spatial filter (Schied et al. 2017, §4.3-4.4) without its temporal part, guided by the pixel-centre primary hit
// (k_denoise_guides, wavefront.cu): base colour, shading normal and hit distance t.
//   k_denoise_prepare   c = accum / samples; demodulated irradiance c / max(albedo, 1e-3); depth gradient of t
//   k_denoise_variance  luminance variance over a 7x7 window weighted by the normal and depth weights
//   k_atrous            one 5x5 B3-spline level with step 2^k, K times, ping-ponging (irradiance.rgb, variance)
// The last level remodulates.  Pixels without a hit or with a non-finite colour ("invalid") keep c and take no part.
// tests/denoise_ref.py is the numpy reference and follows these kernels operation for operation.
#include "core_internal.h"

#include <algorithm>
#include <cmath>

namespace pt
{

namespace
{

constexpr float kAlbedoFloor = 1e-3f; // demodulation divides by max(albedo, kAlbedoFloor) per channel
constexpr float kEpsDepth = 1e-4f;    // w_z denominator offset, in scene units
constexpr float kEpsLuminance = 1e-10f; // w_l denominator offset
constexpr int kVarianceRadius = 3;    // 7x7 variance window

__device__ __forceinline__ float luminance(float r, float g, float b) { return 0.2126f * r + 0.7152f * g + 0.0722f * b; }

// max(0, n_p . n_q)^sigma_n
__device__ __forceinline__ float normalWeight(float4 a, float4 b, float sigmaN)
{
    return powf(fmaxf(0.0f, a.x * b.x + a.y * b.y + a.z * b.z), sigmaN);
}

// exp(-|t_p - t_q| / (sigma_z |grad t_p . (q - p)| + eps)), (dx, dy) = q - p in pixels
__device__ __forceinline__ float depthWeight(float tp, float tq, float2 g, float dx, float dy, float sigmaZ)
{
    return expf(-fabsf(tp - tq) / (sigmaZ * fabsf(g.x * dx + g.y * dy) + kEpsDepth));
}

// one-sided difference of t towards the hit neighbour whose difference is smaller (a depth edge is not a slope); 0 without one
__device__ __forceinline__ float depthSlope(float t, float tb, bool hb, float tf, bool hf)
{
    const float db = t - tb, df = tf - t;
    if (hb && hf)
        return fabsf(df) <= fabsf(db) ? df : db;
    return hf ? df : hb ? db : 0.0f;
}

__global__ void __launch_bounds__(256) k_denoise_prepare(const float4 *__restrict__ accum, float samples, const float4 *__restrict__ albedoT,
                                                         const float4 *__restrict__ normal, uint32_t W, uint32_t H, float4 *__restrict__ nt,
                                                         float4 *__restrict__ irr, float2 *__restrict__ grad, float4 *__restrict__ out)
{
    const uint32_t x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= W || y >= H)
        return;
    const size_t i = (size_t)y * W + x;
    const float4 a = __ldg(accum + i);
    const float cr = a.x / samples, cg = a.y / samples, cb = a.z / samples;
    out[i] = make_float4(cr, cg, cb, 1.0f);
    const float4 g = __ldg(albedoT + i), n = __ldg(normal + i);
    const bool valid = g.w >= 0.0f && isfinite(cr) && isfinite(cg) && isfinite(cb);
    nt[i] = make_float4(n.x, n.y, n.z, valid ? g.w : -1.0f);
    if (!valid)
        return;
    irr[i] = make_float4(cr / fmaxf(g.x, kAlbedoFloor), cg / fmaxf(g.y, kAlbedoFloor), cb / fmaxf(g.z, kAlbedoFloor), 0.0f);
    auto tAt = [&](uint32_t xx, uint32_t yy) { return __ldg(&albedoT[(size_t)yy * W + xx].w); };
    const float tl = x > 0 ? tAt(x - 1, y) : -1.0f, tr = x + 1 < W ? tAt(x + 1, y) : -1.0f;
    const float tu = y > 0 ? tAt(x, y - 1) : -1.0f, td = y + 1 < H ? tAt(x, y + 1) : -1.0f;
    grad[i] = make_float2(depthSlope(g.w, tl, tl >= 0.0f, tr, tr >= 0.0f), depthSlope(g.w, tu, tu >= 0.0f, td, td >= 0.0f));
}

// Variance of the luminance over the 7x7 window around p, each tap weighted by w_n * w_z (the centre by 1); taken about
// l_p, which keeps the moments free of cancellation: var = max(0, m2 - m1^2), m_k = sum w (l_q - l_p)^k / sum w.
__global__ void __launch_bounds__(256) k_denoise_variance(const float4 *__restrict__ irr, const float4 *__restrict__ nt,
                                                          const float2 *__restrict__ grad, uint32_t W, uint32_t H, float sigmaN,
                                                          float sigmaZ, float4 *__restrict__ dst)
{
    const uint32_t x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= W || y >= H)
        return;
    const size_t i = (size_t)y * W + x;
    const float4 np = __ldg(nt + i);
    if (np.w < 0.0f)
        return;
    const float4 ip = __ldg(irr + i);
    const float2 g = __ldg(grad + i);
    const float lp = luminance(ip.x, ip.y, ip.z);
    float sw = 0.0f, s1 = 0.0f, s2 = 0.0f;
    for (int dy = -kVarianceRadius; dy <= kVarianceRadius; dy++)
        for (int dx = -kVarianceRadius; dx <= kVarianceRadius; dx++)
        {
            const int qx = (int)x + dx, qy = (int)y + dy;
            if (qx < 0 || qy < 0 || qx >= (int)W || qy >= (int)H)
                continue;
            const size_t q = (size_t)qy * W + qx;
            const float4 nq = __ldg(nt + q);
            if (nq.w < 0.0f)
                continue;
            const float w = (dx == 0 && dy == 0) ? 1.0f
                                                 : normalWeight(np, nq, sigmaN) * depthWeight(np.w, nq.w, g, (float)dx, (float)dy, sigmaZ);
            const float4 iq = __ldg(irr + q);
            const float d = luminance(iq.x, iq.y, iq.z) - lp;
            sw += w;
            s1 += w * d;
            s2 += w * d * d;
        }
    const float m1 = s1 / sw;
    dst[i] = make_float4(ip.x, ip.y, ip.z, fmaxf(0.0f, s2 / sw - m1 * m1));
}

// One a-trous level (SVGF eq. 1-3 and the variance update of §4.3): 5x5 taps at step 2^k with the B3 spline
// h = (1, 4, 6, 4, 1) / 16 and w = w_n * w_z * w_l (the centre tap w = 1); the luminance scale is the 3x3 Gaussian
// (1, 2, 1)^2 of the variance over valid pixels.  The last level writes mean radiance (irradiance * max(albedo, 1e-3)).
__global__ void __launch_bounds__(256) k_atrous(const float4 *__restrict__ src, const float4 *__restrict__ nt, const float2 *__restrict__ grad,
                                                uint32_t W, uint32_t H, int step, float sigmaL, float sigmaN, float sigmaZ,
                                                float4 *__restrict__ dst, const float4 *__restrict__ albedoT, float4 *__restrict__ out)
{
    const uint32_t x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= W || y >= H)
        return;
    const size_t i = (size_t)y * W + x;
    const float4 np = __ldg(nt + i);
    if (np.w < 0.0f)
        return;
    float sv = 0.0f, sk = 0.0f;
    for (int dy = -1; dy <= 1; dy++)
        for (int dx = -1; dx <= 1; dx++)
        {
            const int qx = (int)x + dx, qy = (int)y + dy;
            if (qx < 0 || qy < 0 || qx >= (int)W || qy >= (int)H)
                continue;
            const size_t q = (size_t)qy * W + qx;
            if (__ldg(&nt[q].w) < 0.0f)
                continue;
            const float k = (float)((2 - abs(dx)) * (2 - abs(dy)));
            sv += k * __ldg(&src[q].w);
            sk += k;
        }
    const float denomL = sigmaL * sqrtf(sv / sk) + kEpsLuminance;
    const float4 ip = __ldg(src + i);
    const float2 g = __ldg(grad + i);
    const float lp = luminance(ip.x, ip.y, ip.z);
    const float h[5] = { 0.0625f, 0.25f, 0.375f, 0.25f, 0.0625f };
    float sr = 0.0f, sg = 0.0f, sb = 0.0f, svar = 0.0f, sw = 0.0f;
#pragma unroll
    for (int dy = -2; dy <= 2; dy++)
#pragma unroll
        for (int dx = -2; dx <= 2; dx++)
        {
            const int qx = (int)x + dx * step, qy = (int)y + dy * step;
            if (qx < 0 || qy < 0 || qx >= (int)W || qy >= (int)H)
                continue;
            const size_t q = (size_t)qy * W + qx;
            const float4 nq = __ldg(nt + q);
            if (nq.w < 0.0f)
                continue;
            const float4 iq = __ldg(src + q);
            float w = 1.0f;
            if (dx != 0 || dy != 0)
                w = normalWeight(np, nq, sigmaN) * depthWeight(np.w, nq.w, g, (float)(dx * step), (float)(dy * step), sigmaZ) *
                    expf(-fabsf(lp - luminance(iq.x, iq.y, iq.z)) / denomL);
            const float hw = h[dx + 2] * h[dy + 2] * w;
            sr += hw * iq.x;
            sg += hw * iq.y;
            sb += hw * iq.z;
            svar += hw * hw * iq.w;
            sw += hw;
        }
    const float r = sr / sw, gg = sg / sw, b = sb / sw;
    if (out)
    {
        const float4 a = __ldg(albedoT + i);
        out[i] = make_float4(r * fmaxf(a.x, kAlbedoFloor), gg * fmaxf(a.y, kAlbedoFloor), b * fmaxf(a.z, kAlbedoFloor), 1.0f);
    }
    else
        dst[i] = make_float4(r, gg, b, svar / (sw * sw));
}

} // namespace

pt_status checkDenoise(Context *ctx, const char *what, const pt_render_params *params, const pt_denoise_params *dn, float divisor,
                       const float *out, size_t outBytes)
{
    if (!params || !dn)
        return fail(ctx, PT_ERR_INVALID_ARGUMENT, what, "NULL argument");
    if (!ctx->hasScene)
        return fail(ctx, PT_ERR_NO_SCENE, what, "no scene uploaded");
    if (!ctx->accum)
        return fail(ctx, PT_ERR_NO_TARGET, what, "pt_render_begin has not been called");
    if (params->lens_radius > 0.0f)
        return fail(ctx, PT_ERR_UNSUPPORTED, what, "lens_radius > 0: pinhole guides cannot describe a defocused image");
    if (divisor == 0.0f)
        return fail(ctx, PT_ERR_INVALID_ARGUMENT, what, "total_samples must be at least 1");
    if (dn->iterations > 8)
        return fail(ctx, PT_ERR_INVALID_ARGUMENT, what, "iterations must be in 0..8");
    for (const float s : { dn->sigma_luminance, dn->sigma_normal, dn->sigma_depth })
        if (!std::isfinite(s) || s < 0.0f)
            return fail(ctx, PT_ERR_INVALID_ARGUMENT, what, "sigmas must be finite and non-negative");
    if (out && outBytes < (size_t)ctx->width * ctx->height * sizeof(float4))
        return fail(ctx, PT_ERR_INVALID_ARGUMENT, what, "output buffer too small");
    return PT_OK;
}

pt_status allocDenoiseBuffers(Context *ctx)
{
    if (ctx->denoised)
        return PT_OK;
    // belongs to the target: freeTarget releases it with the accumulation
    const size_t n = (size_t)ctx->width * ctx->height;
    char *mem = nullptr;
    PT_CUDA_CHECK(ctx, cudaMalloc((void **)&mem, n * (6 * sizeof(float4) + sizeof(float2))));
    ctx->targetAllocs.push_back(mem);
    float4 *f = reinterpret_cast<float4 *>(mem);
    ctx->denoiseAlbedoT = f;
    ctx->denoiseNormal = f + n;
    ctx->denoised = f + 2 * n;
    ctx->denoiseNT = f + 3 * n;
    ctx->denoisePing = f + 4 * n;
    ctx->denoisePong = f + 5 * n;
    ctx->denoiseGrad = reinterpret_cast<float2 *>(f + 6 * n);
    return PT_OK;
}

void launchDenoisePrepare(Context *ctx, const pt_render_params *params, const float4 *src, float divisor)
{
    const uint32_t W = ctx->width, H = ctx->height;
    launchDenoiseGuides(ctx, params, ctx->denoiseAlbedoT, ctx->denoiseNormal);
    const dim3 block(32, 8), grid((W + 31) / 32, (H + 7) / 8);
    k_denoise_prepare<<<grid, block, 0, ctx->stream>>>(src, divisor, ctx->denoiseAlbedoT, ctx->denoiseNormal, W, H, ctx->denoiseNT,
                                                       ctx->denoisePing, ctx->denoiseGrad, ctx->denoised);
}

void launchDenoiseVariance(Context *ctx, const pt_denoise_params *dn)
{
    const uint32_t W = ctx->width, H = ctx->height;
    const dim3 block(32, 8), grid((W + 31) / 32, (H + 7) / 8);
    k_denoise_variance<<<grid, block, 0, ctx->stream>>>(ctx->denoisePing, ctx->denoiseNT, ctx->denoiseGrad, W, H, dn->sigma_normal,
                                                        dn->sigma_depth, ctx->denoisePong);
}

void launchAtrous(Context *ctx, const pt_denoise_params *dn)
{
    const uint32_t W = ctx->width, H = ctx->height;
    const dim3 block(32, 8), grid((W + 31) / 32, (H + 7) / 8);
    const uint32_t K = dn->iterations;
    float4 *a = ctx->denoisePong, *b = ctx->denoisePing;
    for (uint32_t k = 0; k < K; k++)
    {
        const bool last = k + 1 == K;
        k_atrous<<<grid, block, 0, ctx->stream>>>(a, ctx->denoiseNT, ctx->denoiseGrad, W, H, 1 << k, dn->sigma_luminance, dn->sigma_normal,
                                                  dn->sigma_depth, b, ctx->denoiseAlbedoT, last ? ctx->denoised : nullptr);
        std::swap(a, b);
    }
}

pt_status finishDenoise(Context *ctx, const char *what, float *out, uint32_t launches)
{
    cudaStream_t st = ctx->stream;
    cudaError_t err = cudaGetLastError();
    if (err == cudaSuccess && out)
        err = cudaMemcpyAsync(out, ctx->denoised, (size_t)ctx->width * ctx->height * sizeof(float4), cudaMemcpyDeviceToHost, st);
    if (err == cudaSuccess)
        err = cudaStreamSynchronize(st);
    PT_CUDA_CHECK(ctx, err);
    ctx->stats.kernel_launches = launches;
    const pt_status s = checkStackOverflow(ctx, what);
    if (s == PT_OK)
        ctx->denoiseValid = true;
    return s;
}

pt_status denoise(Context *ctx, const char *what, const pt_render_params *params, const pt_denoise_params *dn, const float4 *src,
                  float divisor, float *out, size_t outBytes)
{
    pt_status s = checkDenoise(ctx, what, params, dn, divisor, out, outBytes);
    if (s == PT_OK)
        s = allocDenoiseBuffers(ctx);
    if (s != PT_OK)
        return s;
    ctx->denoiseValid = false;
    launchDenoisePrepare(ctx, params, src, divisor);
    const uint32_t K = dn->iterations;
    if (K > 0)
    {
        launchDenoiseVariance(ctx, dn);
        launchAtrous(ctx, dn);
    }
    return finishDenoise(ctx, what, out, 2 + (K > 0 ? 1 + K : 0));
}

} // namespace pt
