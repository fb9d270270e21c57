// temporal.cu — the denoiser's temporal stage (DESIGN §3j): SVGF's reprojection and accumulation (Schied et al. 2017,
// §4.1-4.2) in front of the unchanged spatial filter of denoise.cu.
//   guides, k_denoise_prepare   as pt_denoise: c, valid, (N, t), demodulated irradiance i (ping), depth gradient
//   k_temporal_reproject        per valid pixel: the history at its position in the previous call's camera, 2x2 bilinear
//                               taps that pass a depth and a normal test; I += a (i - I), (m1, m2) likewise; ping = I
//   k_denoise_variance          the 7x7 estimate on I (pong), then k_temporal_variance: max(0, m2 - m1^2) where n >= 4
//   k_atrous x K                unchanged; the last level remodulates into ctx->denoised
// The history keeps the unfiltered I, so it does not depend on the filter parameters.  tests/temporal_ref.py is the numpy
// reference and follows k_temporal_reproject operation for operation (the library builds with -fmad=false).
#include "core_internal.h"
#include "shading.cuh"

#include <cmath>
#include <cstring>

namespace pt
{

namespace
{

constexpr float kAlbedoFloor = 1e-3f;      // as denoise.cu: remodulation multiplies by max(albedo, kAlbedoFloor)
constexpr float kDepthTolerance = 0.02f;   // a history tap counts when |t_q - |X - O'|| <= kDepthTolerance |X - O'| ...
constexpr float kNormalTolerance = 0.9f;   // ... and n_q . n_p >= kNormalTolerance
constexpr float kMinHistoryWeight = 1e-3f; // below this sum of the counting taps' bilinear weights the history is rejected
constexpr float kMaxHistory = 65535.0f;    // cap of the history length n
constexpr float kMomentsHistory = 4.0f;    // from this history length on, the variance is the temporal one

enum class History : int { None, Identity, Reproject };

__device__ __forceinline__ float luminance(float r, float g, float b) { return 0.2126f * r + 0.7152f * g + 0.0722f * b; }

// mode None: no history (first call, reset); Identity: the camera is bit-identical to the previous call's, every pixel
// reads its own history; Reproject: the history at X = O + t D projected into `prev` by Cramer's rule.
__global__ void __launch_bounds__(256) k_temporal_reproject(CameraMatrices cam, CameraMatrices prev, History mode, uint32_t W, uint32_t H,
                                                            float alpha, float alphaMoments, const float4 *__restrict__ nt,
                                                            const float4 *__restrict__ albedoT, const float4 *__restrict__ prevNT,
                                                            const float4 *__restrict__ histIrr, const float2 *__restrict__ histMoments,
                                                            float4 *__restrict__ irr, float4 *__restrict__ outIrr,
                                                            float2 *__restrict__ outMoments, float4 *__restrict__ out)
{
    const uint32_t x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= W || y >= H)
        return;
    const size_t i = (size_t)y * W + x;
    const float4 np = __ldg(nt + i);
    if (np.w < 0.0f)
    {
        // invalid: k_denoise_prepare wrote c; the zero history keeps the taps of later calls finite
        outIrr[i] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        outMoments[i] = make_float2(0.0f, 0.0f);
        return;
    }
    float sw = 0.0f, sr = 0.0f, sg = 0.0f, sb = 0.0f, sn = 0.0f, s1 = 0.0f, s2 = 0.0f;
    if (mode != History::None)
    {
        const PrimaryRays pr = constructPrimaryRay((float)x, (float)y, (float)W, (float)H, cam, V2(0.5f, 0.5f), V2(0.0f, 0.0f), 0.0f, 0.0f);
        const vec3 X = pr.origin + np.w * pr.direction;
        const vec3 r = X - V3(prev.view[12], prev.view[13], prev.view[14]);
        const float dist = sqrtf(dot(r, r));
        float xp = (float)x, yp = (float)y;
        bool inFront = true;
        if (mode == History::Reproject)
        {
            // the previous camera's ray through NDC (dx, dy) is O' + s V3 (a dx + b dy + c); solve [A B C] (s dx, s dy, s) = r
            const vec3 A = mulPoint(prev.view, prev.proj[0], prev.proj[1], prev.proj[2], 0.0f);
            const vec3 B = mulPoint(prev.view, prev.proj[4], prev.proj[5], prev.proj[6], 0.0f);
            const vec3 C = mulPoint(prev.view, prev.proj[8] + prev.proj[12], prev.proj[9] + prev.proj[13], prev.proj[10] + prev.proj[14], 0.0f);
            const float det = dot(A, cross(B, C));
            const float d1 = dot(r, cross(B, C)), d2 = dot(A, cross(r, C)), d3 = dot(A, cross(B, r));
            inFront = d3 / det > 0.0f;
            xp = (d1 / d3 + 1.0f) * 0.5f * (float)W - 0.5f;
            yp = (d2 / d3 + 1.0f) * 0.5f * (float)H - 0.5f;
        }
        // no tap lies inside the image outside [-1, W) x [-1, H) (this also rejects NaN)
        if (inFront && xp >= -1.0f && xp < (float)W && yp >= -1.0f && yp < (float)H)
        {
            const float fx0 = floorf(xp), fy0 = floorf(yp);
            const int x0 = (int)fx0, y0 = (int)fy0;
            const float fx = xp - fx0, fy = yp - fy0;
#pragma unroll
            for (int k = 0; k < 4; k++)
            {
                const int qx = x0 + (k & 1), qy = y0 + (k >> 1);
                if (qx < 0 || qy < 0 || qx >= (int)W || qy >= (int)H)
                    continue;
                const size_t q = (size_t)qy * W + qx;
                const float4 nq = __ldg(prevNT + q);
                if (!(nq.w >= 0.0f) || !(fabsf(nq.w - dist) <= kDepthTolerance * dist) ||
                    !(nq.x * np.x + nq.y * np.y + nq.z * np.z >= kNormalTolerance))
                    continue;
                const float w = ((k & 1) ? fx : 1.0f - fx) * ((k >> 1) ? fy : 1.0f - fy);
                const float4 h = __ldg(histIrr + q);
                const float2 m = __ldg(histMoments + q);
                sw += w;
                sr += w * h.x;
                sg += w * h.y;
                sb += w * h.z;
                sn += w * h.w;
                s1 += w * m.x;
                s2 += w * m.y;
            }
        }
    }
    float hr = 0.0f, hg = 0.0f, hb = 0.0f, hn = 0.0f, h1 = 0.0f, h2 = 0.0f;
    if (sw >= kMinHistoryWeight)
        hr = sr / sw, hg = sg / sw, hb = sb / sw, hn = sn / sw, h1 = s1 / sw, h2 = s2 / sw;
    const float n = fminf(hn + 1.0f, kMaxHistory);
    const float a = fmaxf(alpha, 1.0f / n), am = fmaxf(alphaMoments, 1.0f / n);
    const float4 c = irr[i];
    const float ir = hr + a * (c.x - hr), ig = hg + a * (c.y - hg), ib = hb + a * (c.z - hb);
    const float l = luminance(c.x, c.y, c.z);
    const float m1 = h1 + am * (l - h1), m2 = h2 + am * (l * l - h2);
    outIrr[i] = make_float4(ir, ig, ib, n);
    outMoments[i] = make_float2(m1, m2);
    irr[i] = make_float4(ir, ig, ib, 0.0f);
    const float4 g = __ldg(albedoT + i);
    out[i] = make_float4(ir * fmaxf(g.x, kAlbedoFloor), ig * fmaxf(g.y, kAlbedoFloor), ib * fmaxf(g.z, kAlbedoFloor), 1.0f);
}

// the temporal variance in place of k_denoise_variance's 7x7 estimate where the history is long enough (invalid: n = 0)
__global__ void __launch_bounds__(256) k_temporal_variance(const float4 *__restrict__ histIrr, const float2 *__restrict__ histMoments,
                                                           uint32_t pixels, float4 *__restrict__ dst)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= pixels || !(__ldg(&histIrr[i].w) >= kMomentsHistory))
        return;
    const float2 m = __ldg(histMoments + i);
    dst[i].w = fmaxf(0.0f, m.y - m.x * m.x);
}

} // namespace

pt_status denoiseTemporal(Context *ctx, const pt_render_params *params, const pt_denoise_params *dn, const pt_temporal_params *tp,
                          uint32_t totalSamples, float *out, size_t outBytes)
{
    const char *what = "pt_denoise_temporal";
    if (!tp)
        return fail(ctx, PT_ERR_INVALID_ARGUMENT, what, "NULL argument");
    pt_status s = checkDenoise(ctx, what, params, dn, (float)totalSamples, out, outBytes);
    if (s != PT_OK)
        return s;
    if (!(tp->alpha >= 0.0f && tp->alpha <= 1.0f) || !(tp->alpha_moments >= 0.0f && tp->alpha_moments <= 1.0f))
        return fail(ctx, PT_ERR_INVALID_ARGUMENT, what, "alpha and alpha_moments must be in [0, 1]");
    if (ctx->targetContent == Context::TargetContent::Adaptive)
        return fail(ctx, PT_ERR_INVALID_ARGUMENT, what, "the target holds an adaptive render");
    s = allocDenoiseBuffers(ctx);
    if (s != PT_OK)
        return s;
    const uint32_t W = ctx->width, H = ctx->height;
    const size_t n = (size_t)W * H;
    if (!ctx->temporalPrevNT)
    {
        // belongs to the target: freeTarget releases it with the accumulation
        char *mem = nullptr;
        PT_CUDA_CHECK(ctx, cudaMalloc((void **)&mem, n * (3 * sizeof(float4) + 2 * sizeof(float2))));
        ctx->targetAllocs.push_back(mem);
        float4 *f = reinterpret_cast<float4 *>(mem);
        ctx->temporalIrr[0] = f;
        ctx->temporalIrr[1] = f + n;
        ctx->temporalPrevNT = f + 2 * n;
        ctx->temporalMoments[0] = reinterpret_cast<float2 *>(f + 3 * n);
        ctx->temporalMoments[1] = ctx->temporalMoments[0] + n;
        ctx->temporalValid = false;
    }
    ctx->denoiseValid = false;
    CameraMatrices cam, prev;
    std::memcpy(cam.view, params->view_inverse, sizeof(cam.view));
    std::memcpy(cam.proj, params->proj_inverse, sizeof(cam.proj));
    std::memcpy(prev.view, ctx->temporalPrevView, sizeof(prev.view));
    std::memcpy(prev.proj, ctx->temporalPrevProj, sizeof(prev.proj));
    History mode = History::None;
    if (ctx->temporalValid && !tp->reset)
        mode = std::memcmp(&cam, &prev, sizeof(cam)) == 0 ? History::Identity : History::Reproject;

    cudaStream_t st = ctx->stream;
    launchDenoisePrepare(ctx, params, ctx->accum, (float)totalSamples);
    const uint32_t cur = ctx->temporalCurrent, next = cur ^ 1u;
    const dim3 block(32, 8), grid((W + 31) / 32, (H + 7) / 8);
    k_temporal_reproject<<<grid, block, 0, st>>>(cam, prev, mode, W, H, tp->alpha, tp->alpha_moments, ctx->denoiseNT, ctx->denoiseAlbedoT,
                                                  ctx->temporalPrevNT, ctx->temporalIrr[cur], ctx->temporalMoments[cur], ctx->denoisePing,
                                                  ctx->temporalIrr[next], ctx->temporalMoments[next], ctx->denoised);
    const uint32_t K = dn->iterations;
    if (K > 0)
    {
        launchDenoiseVariance(ctx, dn);
        k_temporal_variance<<<(uint32_t)((n + 255) / 256), 256, 0, st>>>(ctx->temporalIrr[next], ctx->temporalMoments[next], (uint32_t)n,
                                                                          ctx->denoisePong);
        launchAtrous(ctx, dn);
    }
    // the next call's previous taps; pt_denoise between two temporal calls rewrites denoiseNT but not this copy
    const cudaError_t err = cudaMemcpyAsync(ctx->temporalPrevNT, ctx->denoiseNT, n * sizeof(float4), cudaMemcpyDeviceToDevice, st);
    ctx->temporalCurrent = next;
    std::memcpy(ctx->temporalPrevView, cam.view, sizeof(cam.view));
    std::memcpy(ctx->temporalPrevProj, cam.proj, sizeof(cam.proj));
    ctx->temporalValid = false;
    PT_CUDA_CHECK(ctx, err);
    s = finishDenoise(ctx, what, out, 3 + (K > 0 ? 2 + K : 0));
    ctx->temporalValid = s == PT_OK;
    return s;
}

pt_status temporalHistory(Context *ctx, float *outIrradianceN, float *outMoments, size_t pixels)
{
    const char *what = "pt_denoise_temporal_history";
    if (!ctx->accum)
        return fail(ctx, PT_ERR_NO_TARGET, what, "pt_render_begin has not been called");
    if (!ctx->temporalValid)
        return fail(ctx, PT_ERR_INVALID_ARGUMENT, what, "no history: no pt_denoise_temporal since the target or the scene changed");
    const size_t n = (size_t)ctx->width * ctx->height;
    if (pixels < n)
        return fail(ctx, PT_ERR_INVALID_ARGUMENT, what, "output buffer too small");
    const uint32_t cur = ctx->temporalCurrent;
    if (outIrradianceN)
        PT_CUDA_CHECK(ctx, cudaMemcpyAsync(outIrradianceN, ctx->temporalIrr[cur], n * sizeof(float4), cudaMemcpyDeviceToHost, ctx->stream));
    if (outMoments)
        PT_CUDA_CHECK(ctx, cudaMemcpyAsync(outMoments, ctx->temporalMoments[cur], n * sizeof(float2), cudaMemcpyDeviceToHost, ctx->stream));
    PT_CUDA_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    return PT_OK;
}

} // namespace pt
