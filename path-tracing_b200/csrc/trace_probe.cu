// trace_probe.cu — pt_test_trace: host rays through the traversal of the render's trace kernels.
//
// k_extend / k_shadow trace through tracePersistent (dynamic ray fetch, deferred commits, straggler splitting); the
// standalone queries run the per-thread traverse().  k_test_trace runs either on caller rays, with the Traverser
// instantiation of k_extend (closest) / k_shadow (occlusion), so that the two can be compared hit for hit.
//
// It lives in a translation unit of its own: added to wavefront.cu it changed the register allocation of the hot
// kernels there (same PTX up to symbol names, different SASS), and the probe must not change what it probes.  The
// launch bounds and the resident grid come from core_internal.h, shared with the render.
#include "core_internal.h"
#include "traverse.cuh"

#include <algorithm>
#include <cstdio>
#include <cstring>

namespace pt
{

namespace
{

// wavefront.cu's toPtHit: leaf-order hit -> (instance, geometry, primitive, t, u, v)
__device__ __forceinline__ pt_hit probeHit(const DeviceScene &s, const Hit &h)
{
    pt_hit r;
    if (h.tri == 0xffffffffu)
    {
        r.instance = r.geometry = r.primitive = PT_NO_HIT;
        r.t = r.u = r.v = 0.0f;
        return r;
    }
    const float4 a8 = __ldg(&s.triShade[__float_as_uint(__ldg(s.triPos + 3 * (size_t)h.tri).w)].a[8]);
    r.instance = __float_as_uint(a8.y);
    r.geometry = __float_as_uint(a8.z);
    r.primitive = __float_as_uint(a8.w);
    r.t = h.t;
    r.u = h.b1;
    r.v = h.b2;
    return r;
}

// decals (may be NULL): r, g, b, a, dist per ray, dist = -1 for none
template <bool CLOSEST, bool ALPHA, bool STATS>
__global__ void __launch_bounds__(128, PT_TRACE_MIN_BLOCKS)
    k_test_trace(DeviceScene s, const pt_ray *rays, uint32_t n, uint32_t persistent, float tmin, uint32_t *workCounter,
                 pt_hit *out, float *decals, TailStats tail)
{
    auto store = [&](uint32_t i, const Hit &hit, const Decal &decal) {
        out[i] = probeHit(s, hit);
        if (decals)
        {
            const bool has = CLOSEST && ALPHA;
            float *d = decals + 5 * (size_t)i;
            d[0] = has ? decal.r : 0.0f, d[1] = has ? decal.g : 0.0f, d[2] = has ? decal.b : 0.0f;
            d[3] = has ? decal.a : 0.0f, d[4] = has ? decal.dist : -1.0f;
        }
    };
    if (!persistent)
    {
        const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
        if (i >= n)
            return;
        const pt_ray r = rays[i];
        Hit hit;
        Decal decal;
        TraversalStats st = { 0, 0, 0 };
        traverse<CLOSEST, ALPHA, STATS>(s, V3(r.origin[0], r.origin[1], r.origin[2]),
                                        V3(r.direction[0], r.direction[1], r.direction[2]), tmin, r.tmax, hit, decal, st);
        store(i, hit, decal);
        return;
    }
    unsigned long long stack[PT_STACK_SIZE];
    Traverser<CLOSEST, ALPHA, STATS> tr;
    tr.stack = stack;
    tr.st = TraversalStats { 0, 0, 0 };
    tracePersistent(
        s, n, workCounter, tr, tmin, [&](uint32_t i) { return i; },
        [&](uint32_t i) {
            const pt_ray r = rays[i];
            RayPacket p;
            p.slot = i;
            p.ox = r.origin[0], p.oy = r.origin[1], p.oz = r.origin[2];
            p.dx = r.direction[0], p.dy = r.direction[1], p.dz = r.direction[2];
            p.tmax = r.tmax;
            return p;
        },
        [&](Traverser<CLOSEST, ALPHA, STATS> &t, uint32_t i) { store(i, t.hit, t.decal); }, tail);
}

} // namespace

pt_status testTrace(Context *ctx, const pt_ray *rays, uint64_t n, uint32_t flags, uint32_t blocks, pt_hit *out, float *outDecals,
                    uint64_t *outTail)
{
    if ((n && (!rays || !out)) || n > (1u << 30) ||
        (flags & ~(uint32_t)(PT_TEST_TRACE_OCCLUSION | PT_TEST_TRACE_PERSISTENT | PT_TEST_TRACE_STATS)))
        return fail(ctx, PT_ERR_INVALID_ARGUMENT, "pt_test_trace", "bad argument");
    if (!ctx->hasScene)
        return fail(ctx, PT_ERR_NO_SCENE, "pt_test_trace", "no scene uploaded");
    // tracePersistent traces every ray of a launch with one tmin
    for (uint64_t i = 1; i < n; i++)
        if (!(rays[i].tmin == rays[0].tmin))
            return fail(ctx, PT_ERR_INVALID_ARGUMENT, "pt_test_trace", "the rays' tmin values differ");
    if (outTail)
        std::memset(outTail, 0, 4 * sizeof(uint64_t));
    if (n == 0)
        return PT_OK;
    const bool closest = !(flags & PT_TEST_TRACE_OCCLUSION), persistent = (flags & PT_TEST_TRACE_PERSISTENT) != 0;
    const bool stats = (flags & PT_TEST_TRACE_STATS) != 0, alpha = ctx->scene.hasAlpha != 0;
    pt_ray *dRays = nullptr;
    pt_hit *dOut = nullptr;
    float *dDecals = nullptr;
    unsigned long long *dTail = nullptr; // visit histogram [8], warp iterations, drain iterations, max drain iterations
    uint32_t *dWork = nullptr;           // behind them: the ray-queue position counter
    const size_t tailBytes = 11 * sizeof(unsigned long long) + sizeof(uint32_t);
    PT_CUDA_CHECK(ctx, cudaMalloc((void **)&dRays, n * sizeof(pt_ray)));
    cudaError_t err = cudaMalloc((void **)&dOut, n * sizeof(pt_hit));
    if (err == cudaSuccess && outDecals)
        err = cudaMalloc((void **)&dDecals, n * 5 * sizeof(float));
    if (err == cudaSuccess)
        err = cudaMalloc((void **)&dTail, tailBytes);
    if (err == cudaSuccess)
    {
        dWork = reinterpret_cast<uint32_t *>(dTail + 11);
        err = cudaMemsetAsync(dTail, 0, tailBytes, ctx->stream);
    }
    if (err == cudaSuccess)
        err = cudaMemcpyAsync(dRays, rays, n * sizeof(pt_ray), cudaMemcpyHostToDevice, ctx->stream);
    if (err == cudaSuccess)
    {
        const TailStats tail { dTail, dTail + 8, dTail + 9, dTail + 10 };
        auto launch = [&](auto kernel) {
            uint32_t grid = (uint32_t)((n + 127) / 128);
            if (persistent && blocks)
                grid = std::min(grid, blocks);
            else if (persistent)
                grid = residentTraceGrid(ctx, kernel, (uint32_t)n); // the grid of the render's trace launches
            kernel<<<grid, 128, 0, ctx->stream>>>(ctx->scene, dRays, (uint32_t)n, persistent ? 1u : 0u, rays[0].tmin, dWork, dOut,
                                                  dDecals, tail);
        };
#define PT_TEST_TRACE_LAUNCH(C, A) (stats ? launch(k_test_trace<C, A, true>) : launch(k_test_trace<C, A, false>))
        if (closest)
            alpha ? PT_TEST_TRACE_LAUNCH(true, true) : PT_TEST_TRACE_LAUNCH(true, false);
        else
            alpha ? PT_TEST_TRACE_LAUNCH(false, true) : PT_TEST_TRACE_LAUNCH(false, false);
#undef PT_TEST_TRACE_LAUNCH
        err = cudaGetLastError();
    }
    if (err == cudaSuccess)
        err = cudaMemcpyAsync(out, dOut, n * sizeof(pt_hit), cudaMemcpyDeviceToHost, ctx->stream);
    if (err == cudaSuccess && outDecals)
        err = cudaMemcpyAsync(outDecals, dDecals, n * 5 * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream);
    unsigned long long tailHost[11] = {};
    if (err == cudaSuccess)
        err = cudaMemcpyAsync(tailHost, dTail, sizeof(tailHost), cudaMemcpyDeviceToHost, ctx->stream);
    if (err == cudaSuccess)
        err = cudaStreamSynchronize(ctx->stream);
    // this translation unit's own overflow counter (g_stackOverflows is static: one per unit)
    unsigned int overflows = 0;
    if (err == cudaSuccess)
        err = cudaMemcpyFromSymbol(&overflows, g_stackOverflows, sizeof(overflows));
    cudaFree(dRays);
    cudaFree(dOut);
    cudaFree(dDecals);
    cudaFree(dTail);
    PT_CUDA_CHECK(ctx, err);
    if (outTail)
    {
        outTail[0] = tailHost[8];
        outTail[1] = tailHost[9];
        outTail[2] = tailHost[10];
        outTail[3] = overflows;
    }
    if (overflows == 0)
        return PT_OK;
    const unsigned int zero = 0;
    cudaMemcpyToSymbol(g_stackOverflows, &zero, sizeof(zero));
    ctx->stats.stack_overflows = overflows;
    char buf[192];
    std::snprintf(buf, sizeof(buf), "the traversal stack (%d entries) overflowed %u times on a BVH of depth %u: sub-trees were "
                                    "skipped, the result is not valid", PT_STACK_SIZE, overflows, ctx->bvhMaxDepth);
    return fail(ctx, PT_ERR_UNSUPPORTED, "pt_test_trace", buf);
}

} // namespace pt
