// emitters.cu — the emitter table of PT_LIGHT_SAMPLING_EMISSIVE_MIS (DESIGN.md §3g; an extension, no GLSL counterpart).
//
// k_emitters finds the emissive triangles and their power, area x luminance of the emission averaged over the triangle;
// the host quantises the powers to integer weights and builds a Walker / Vose alias table from them with integer
// arithmetic in a fixed order, so the table is exact and the same on every GPU and in the CPU reference
// (tests/emissive_oracle.cpp buildEmitterTable, same definitions); k_emitter_records gathers the 64-byte records k_shade_emissive samples points from.
// Built at the first render in the mode after an upload, an update that moves geometry, a texture upload or a sampler change.
#include "core_internal.h"
#include "shading.cuh"

#include <algorithm>
#include <cmath>

namespace pt
{

namespace
{

// One thread per BVH reference: every reference of a triangle carries the same corners, so the (identical) writes of a
// triangle's references are equivalent.  Only opaque geometry emits in NEE: any-hit drops the transparent texels of
// alpha-tested geometry, which BSDF rays therefore never see.
__global__ void k_emitters(DeviceScene s, float2 *__restrict__ areaPower, uint32_t *__restrict__ refOf)
{
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= s.triCount)
        return;
    const float4 q0 = __ldg(s.triPos + 3 * (size_t)k), q1 = __ldg(s.triPos + 3 * (size_t)k + 1);
    const float4 q2 = __ldg(s.triPos + 3 * (size_t)k + 2);
    float4 e;
    uint32_t slot;
    if (!(__float_as_uint(q1.w) & PT_TRI_FLAG_OPAQUE) || !emissiveSource(s, __float_as_uint(q2.w), e, slot))
        return;
    const uint32_t flat = __float_as_uint(q0.w);
    const TriShade &ts = s.triShade[flat];
    const float4 a6 = __ldg(&ts.a[6]), a7 = __ldg(&ts.a[7]), a8 = __ldg(&ts.a[8]);
    const vec3 c = cross(V3(q1) - V3(q0), V3(q2) - V3(q0));
    const float area = 0.5f * sqrtf(dot(c, c));
    // one textureGrad fetch at the UV centroid with the triangle's UV extent as footprint: about the triangle's average
    const float u0 = a6.w, v0 = a7.x, u1 = a7.y, v1 = a7.z, u2 = a7.w, v2 = a8.x;
    const float u = (u0 + u1 + u2) / 3.0f, v = (v0 + v1 + v2) / 3.0f;
    const float du = fmaxf(u0, fmaxf(u1, u2)) - fminf(u0, fminf(u1, u2));
    const float dv = fmaxf(v0, fmaxf(v1, v2)) - fminf(v0, fminf(v1, v2));
    const float4 t = textureGrad(s, slot, u, v, make_float4(du, 0.0f, 0.0f, dv));
    const vec3 E = (V3(t) + V3(e)) * e.w;
    const float luminance = 0.2126f * E.x + 0.7152f * E.y + 0.0722f * E.z;
    areaPower[flat] = make_float2(area, area * fmaxf(luminance, 0.0f));
    refOf[flat] = k;
}

__global__ void k_emitter_records(DeviceScene s, const uint32_t *__restrict__ ids, const uint32_t *__restrict__ refOf, uint32_t n,
                                  float4 *__restrict__ rec)
{
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n)
        return;
    const uint32_t flat = ids[k], r = refOf[flat];
    const float4 q0 = __ldg(s.triPos + 3 * (size_t)r), q1 = __ldg(s.triPos + 3 * (size_t)r + 1);
    const float4 q2 = __ldg(s.triPos + 3 * (size_t)r + 2);
    const TriShade &ts = s.triShade[flat];
    const float4 a6 = __ldg(&ts.a[6]), a7 = __ldg(&ts.a[7]), a8 = __ldg(&ts.a[8]);
    rec[4 * (size_t)k + 0] = make_float4(q0.x, q0.y, q0.z, q1.x);
    rec[4 * (size_t)k + 1] = make_float4(q1.y, q1.z, q2.x, q2.y);
    rec[4 * (size_t)k + 2] = make_float4(q2.z, a6.w, a7.x, a7.y);
    rec[4 * (size_t)k + 3] = make_float4(a7.z, a7.w, a8.x, q2.w);
}

template <typename T> cudaError_t allocCopy(Context *ctx, T **out, const T *src, size_t n)
{
    cudaError_t err = cudaMalloc((void **)out, std::max<size_t>(n, 1) * sizeof(T));
    if (err != cudaSuccess)
        return err;
    ctx->emitterAllocs.push_back(*out);
    return n ? cudaMemcpyAsync(*out, src, n * sizeof(T), cudaMemcpyHostToDevice, ctx->stream) : cudaSuccess;
}

} // namespace

// Integer weights and the alias table (DESIGN.md §3g).  w = max(1, rint(power / maxPower x 2^24)); bucket k of n keeps k
// with probability s_k / W, where s_k is its share of n x w in units of W = sum(w), and hands the rest to its alias.
// Vose's pairing with both work lists filled in index order and used as stacks: small (s < W) and large (s >= W).
// The probability is stored as a 32-bit fraction x < threshold; a full bucket is its own alias with threshold 2^32 - 1.
void buildAliasTable(const std::vector<float> &power, std::vector<uint32_t> &weights, std::vector<uint2> &alias)
{
    const size_t n = power.size();
    float maxPower = 0.0f;
    for (float p : power)
        maxPower = std::max(maxPower, p);
    weights.resize(n);
    alias.resize(n);
    uint64_t W = 0;
    for (size_t k = 0; k < n; k++)
    {
        weights[k] = std::max<uint32_t>(1u, (uint32_t)std::rint((double)power[k] / (double)maxPower * 16777216.0));
        W += weights[k];
    }
    std::vector<uint64_t> share(n);
    std::vector<uint32_t> small, large;
    for (size_t k = 0; k < n; k++)
    {
        share[k] = (uint64_t)weights[k] * n;
        (share[k] < W ? small : large).push_back((uint32_t)k);
    }
    while (!small.empty() && !large.empty())
    {
        const uint32_t l = small.back(), g = large.back();
        small.pop_back();
        alias[l] = make_uint2((uint32_t)(((unsigned __int128)share[l] << 32) / W), g);
        share[g] -= W - share[l];
        if (share[g] < W)
        {
            large.pop_back();
            small.push_back(g);
        }
    }
    for (uint32_t k : small)
        alias[k] = make_uint2(0xffffffffu, k);
    for (uint32_t k : large)
        alias[k] = make_uint2(0xffffffffu, k);
}

void freeEmitters(Context *ctx)
{
    if (!ctx->emitterAllocs.empty() && ctx->stream)
        cudaStreamSynchronize(ctx->stream);
    for (void *p : ctx->emitterAllocs)
        cudaFree(p);
    ctx->emitterAllocs.clear();
    ctx->emitters = EmitterTable {};
    ctx->emitterIds.clear();
    ctx->emitterWeights.clear();
    ctx->emitterAlias.clear();
    ctx->emittersValid = false;
}

pt_status buildEmitters(Context *ctx)
{
    freeEmitters(ctx);
    const DeviceScene &s = ctx->scene;
    const uint32_t flatCount = s.triCount ? (uint32_t)ctx->triangleCount : 0u;
    ScopedEvent ev0, ev1;
    cudaEventRecord(ev0, ctx->stream);
    // per flat triangle (area, power) and one of its BVH references: freed on every path out of this function
    struct Temp
    {
        float2 *areaPower = nullptr;
        uint32_t *ref = nullptr;
        ~Temp()
        {
            cudaFree(areaPower);
            cudaFree(ref);
        }
    } temp;
    PT_CUDA_CHECK(ctx, cudaMalloc((void **)&temp.areaPower, std::max(flatCount, 1u) * sizeof(float2)));
    PT_CUDA_CHECK(ctx, cudaMalloc((void **)&temp.ref, std::max(flatCount, 1u) * sizeof(uint32_t)));
    float2 *dAreaPower = temp.areaPower;
    const uint32_t *dRef = temp.ref;
    PT_CUDA_CHECK(ctx, cudaMemsetAsync(dAreaPower, 0, std::max(flatCount, 1u) * sizeof(float2), ctx->stream));
    if (s.triCount)
        k_emitters<<<(s.triCount + 255) / 256, 256, 0, ctx->stream>>>(s, dAreaPower, temp.ref);
    std::vector<float2> areaPower(flatCount);
    if (flatCount)
        PT_CUDA_CHECK(ctx, cudaMemcpyAsync(areaPower.data(), dAreaPower, flatCount * sizeof(float2), cudaMemcpyDeviceToHost, ctx->stream));
    PT_CUDA_CHECK(ctx, cudaStreamSynchronize(ctx->stream));

    // emitters in flat order: a finite, positive power (degenerate and black-emitting triangles are never sampled)
    std::vector<float> power;
    for (uint32_t f = 0; f < flatCount; f++)
        if (std::isfinite(areaPower[f].y) && areaPower[f].y > 0.0f)
        {
            ctx->emitterIds.push_back(f);
            power.push_back(areaPower[f].y);
        }
    buildAliasTable(power, ctx->emitterWeights, ctx->emitterAlias);
    const uint32_t n = (uint32_t)power.size();
    uint64_t W = 0;
    for (uint32_t w : ctx->emitterWeights)
        W += w;
    std::vector<float> emitterPdf(n), pdfOverArea(n ? flatCount : 0, 0.0f);
    for (uint32_t k = 0; k < n; k++)
    {
        const uint32_t f = ctx->emitterIds[k];
        emitterPdf[k] = (float)((double)ctx->emitterWeights[k] / (double)W / (double)areaPower[f].x);
        pdfOverArea[f] = emitterPdf[k];
    }

    EmitterTable &t = ctx->emitters;
    t.count = n;
    if (n)
    {
        uint32_t *dIds;
        uint2 *dAlias;
        float *dEmitterPdf, *dPdfOverArea;
        float4 *dRec;
        PT_CUDA_CHECK(ctx, allocCopy(ctx, &dIds, ctx->emitterIds.data(), n));
        PT_CUDA_CHECK(ctx, allocCopy(ctx, &dAlias, ctx->emitterAlias.data(), n));
        PT_CUDA_CHECK(ctx, allocCopy(ctx, &dEmitterPdf, emitterPdf.data(), n));
        PT_CUDA_CHECK(ctx, allocCopy(ctx, &dPdfOverArea, pdfOverArea.data(), flatCount));
        PT_CUDA_CHECK(ctx, cudaMalloc((void **)&dRec, (size_t)n * 4 * sizeof(float4)));
        ctx->emitterAllocs.push_back(dRec);
        k_emitter_records<<<(n + 255) / 256, 256, 0, ctx->stream>>>(s, dIds, dRef, n, dRec);
        t.rec = dRec;
        t.alias = dAlias;
        t.emitterPdf = dEmitterPdf;
        t.pdfOverArea = dPdfOverArea;
    }
    cudaEventRecord(ev1, ctx->stream);
    PT_CUDA_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    PT_CUDA_CHECK(ctx, cudaGetLastError());
    cudaEventElapsedTime(&ctx->emitterBuildMs, ev0, ev1);
    ctx->emittersValid = true;
    return PT_OK;
}

} // namespace pt
