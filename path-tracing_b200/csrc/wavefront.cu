// wavefront.cu — the path-tracing hot path as wavefront kernels for sm_100a.
//
// A fixed pool of path SLOTS pulls WORK ITEMS (pixel, sample) from a global counter, in
// sample-major order, so the wavefront stays full until the very last items of a round
// regardless of how path lengths differ between pixels.  A finished path parks its radiance in
// the round's sample buffer sbuf[sample][pixel]; k_resolve then adds the samples of every pixel
// to the accumulation image IN SAMPLE ORDER, which is the reference's summation order
// (raygen.rgen:115-117 runs once per frame with SampleCount = 1) — so the image does not depend
// on scheduling, slot count or tile partition, bit for bit.  Per iteration:
//
//   k_extend   closest-hit traversal of every active slot's ray          (raygen.rgen:68)
//              PATH REGENERATION happens here too: a slot whose path ended in the previous
//              iteration (regen queue) is finished while its ray would be fetched — miss.rmiss,
//              NaN/Inf restart or park the sample and pull the next work item, generate the primary
//              ray (raygen.rgen:38-58, 71-75, 99-117) — and the new ray is traversed right away
//   k_shade    closestHit.rchit + the raygen bounce logic                  (raygen.rgen:76-96)
//              emits a shadow ray into a compacted queue when NEE can contribute
//   k_shadow   occlusion traversal, adds the direct-light contribution    (raygen.rgen:79-81)
//
// Path state is one 256-byte record per slot (core_internal.h); queues hold slot indices and are
// compacted with warp-aggregated atomics.  Continuing (incoherent) paths and ended paths (whose
// successors are coherent primary rays: consecutive pixels of an 8x4 block) go to separate queues
// so that warps of k_extend are not a mix of both.  Queue order never influences a slot's
// arithmetic, so results are deterministic.
#include "core_internal.h"
#include "shading.cuh"
#include "traverse.cuh"

#include <cub/device/device_radix_sort.cuh>

#include <algorithm>
#include <cstdlib>
#include <cstring>

namespace pt
{

namespace
{

// resident 128-thread blocks per SM the register allocation must allow (tuned on the B200, see DESIGN.md)
#ifndef PT_TRACE_MIN_BLOCKS
#define PT_TRACE_MIN_BLOCKS 8
#endif
// bits of the leaf-order triangle index the hit queue is sorted by; one more bit sends unused entries
// to the end, and CUB's onesweep sort takes one pass per 8 bits: 15 + 1 = two passes
#ifndef PT_HIT_KEY_BITS
#define PT_HIT_KEY_BITS 15
#endif
#ifndef PT_SHADE_MIN_BLOCKS
#define PT_SHADE_MIN_BLOCKS 4
#endif

#ifndef PT_SHADE_GRID_PER_SM
#define PT_SHADE_GRID_PER_SM 4 // k_shade blocks per SM = the resident ones (grid-stride loop over the hits).  Measured 4 / 8 / 16 / 64: alone the kernel
                               // likes MORE blocks (chess 55.2 / 54.3 / 53.4 / 50.2 ms), the two overlapping pools fewer (2368 / 2360 / 2352 / 2341 Mrays/s)
#endif

constexpr uint32_t kMaxRestarts = 1024; // the reference's restart loop is unbounded; see oracle
// path state word (PathRecord::thr.w): bounce [0, 8), NaN/Inf restarts of the frame [8, 19), sample of the frame [19, 32)
constexpr uint32_t kRestartShift = 8, kRestartMask = 0x7ffu, kSampleShift = 19;
constexpr uint32_t kMaxSamplesPerFrame = 1u << (32 - kSampleShift);

struct RenderConst
{
    DeviceScene scene;
    PathState ps;
    CameraMatrices cam;
    float4 *accum;
    DeviceCounters *counters;
    QueueCounts *qc;
    uint32_t width, height;
    uint32_t firstSample, sampleCount;
    uint32_t samplesPerFrame;    // raygen.rgen's SampleCount: samples one work item (pixel, frame) runs on ONE rng stream
    uint32_t bounceCount;
    float lensRadius, focalDistance;
    uint32_t missFlags, hitFlags;
    uint32_t slotBase;           // first slot of this pool
    uint32_t slotCount;          // slots of this pool in use
    uint32_t *nextItem;          // next work item of the round (shared by all pools)
    const uint32_t *pixelList;   // pixels of the tile set in 8x4-block order
    uint32_t pixelCount;
    float4 *sbuf;                // [roundSamples][pixelCount] radiance of the finished samples of the round
    uint32_t roundBase;          // first sample of the round, relative to firstSample
    uint32_t roundSamples;
    uint32_t itemCount;          // roundSamples * pixelCount; item = sample * pixelCount + pixel-list index
    uint32_t hitKeyShift;        // hit sort key = leaf-order triangle index >> hitKeyShift
    uint32_t sortHits;           // k_shade reads hitQSorted instead of hitQ
};

__device__ __forceinline__ uint32_t laneId() { return threadIdx.x & 31u; }

// warp-aggregated atomic increment (all currently converged lanes that call it share one atomic)
__device__ __forceinline__ uint32_t atomicAggInc(uint32_t *counter)
{
    const unsigned mask = __activemask();
    const int leader = __ffs(mask) - 1;
    uint32_t base = 0;
    if ((int)laneId() == leader)
        base = atomicAdd(counter, (uint32_t)__popc(mask));
    base = __shfl_sync(mask, base, leader);
    return base + __popc(mask & ((1u << laneId()) - 1u));
}

__device__ __forceinline__ void warpAdd(unsigned long long *counter, uint32_t value)
{
    for (int o = 16; o > 0; o >>= 1)
        value += __shfl_down_sync(0xffffffffu, value, o);
    if (laneId() == 0 && value)
        atomicAdd(counter, (unsigned long long)value);
}

// queue entry flags (slot indices need 24 bits at most)
constexpr uint32_t kRegen = 0x40000000u;     // regen queue entry: the slot's path has ended
constexpr uint32_t kRegenMiss = 0x80000000u; // ... by leaving the scene: throughput * sky is still to be added
constexpr uint32_t kSlotMask = 0x3fffffffu;
constexpr uint32_t kDeadSlot = 0xffffffffu;  // RayPacket::slot of a regen entry that found no work item left

// ---------------------------------------------------------------------------------------------
// raygen.rgen:44-60 — start one sample of a slot's pixel; returns the primary ray
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ PrimaryRays generatePath(const RenderConst &rc, uint32_t slot, uint32_t pixel, uint32_t item,
                                                    uint32_t rng, uint32_t restarts, uint32_t smpl = 0, vec3 radiance = { 0.0f, 0.0f, 0.0f })
{
    const uint32_t py = pixel / rc.width, px = pixel - py * rc.width;
    const float ux = rnd(rng);
    const float uy = rnd(rng);
    vec2 u2 = V2(0.0f, 0.0f);
    if (rc.lensRadius > 0)
    {
        u2.x = rnd(rng);
        u2.y = rnd(rng);
    }
    const PrimaryRays pr = constructPrimaryRay((float)px, (float)py, (float)rc.width, (float)rc.height, rc.cam, V2(ux, uy),
                                               u2, rc.lensRadius, rc.focalDistance);
    PathRecord &rec = rc.ps.rec[slot];
    rec.rayO = make_float4(pr.origin.x, pr.origin.y, pr.origin.z, 0.0f); // MaxRoughness = 0
    rec.rayD = make_float4(pr.direction.x, pr.direction.y, pr.direction.z, __uint_as_float(rng));
    rec.thr = make_float4(1.0f, 1.0f, 1.0f, __uint_as_float((smpl << kSampleShift) | (restarts << kRestartShift))); // bounce 0
    rec.rad = make_float4(radiance.x, radiance.y, radiance.z, __uint_as_float(item));
    rec.diff0 = make_float4(pr.origin.x, pr.origin.y, pr.origin.z, pr.rxDirection.x);
    rec.diff1 = make_float4(pr.rxDirection.y, pr.rxDirection.z, pr.origin.x, pr.origin.y);
    rec.diff2 = make_float4(pr.origin.z, pr.ryDirection.x, pr.ryDirection.y, pr.ryDirection.z);
    return pr;
}

// work item -> (pixel, absolute sample index); starts the item's path in `slot`
__device__ __forceinline__ PrimaryRays startItem(const RenderConst &rc, uint32_t slot, uint32_t item)
{
    const uint32_t s = item / rc.pixelCount, pi = item - s * rc.pixelCount;
    const uint32_t pixel = __ldg(rc.pixelList + pi);
    const uint32_t py = pixel / rc.width, px = pixel - py * rc.width;
    // frame s of the round: TotalSamples = samples accumulated before it (Renderer.cpp:1694-1700)
    return generatePath(rc, slot, pixel, item, initRng(px, py, rc.width, rc.firstSample + (rc.roundBase + s) * rc.samplesPerFrame), 0);
}

// slot i (of all pools together) starts with work item i of the round
__global__ void __launch_bounds__(256) k_init(RenderConst rc)
{
    const uint32_t stride = gridDim.x * blockDim.x;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < rc.slotCount; i += stride)
    {
        const uint32_t slot = rc.slotBase + i;
        rc.ps.contQ[0][i] = slot;
        startItem(rc, slot, slot);
    }
    if (blockIdx.x == 0 && threadIdx.x == 0)
    {
        rc.qc->cont[0] = rc.slotCount;
        rc.qc->regen[0] = 0;
        rc.qc->cont[1] = 0;
        rc.qc->regen[1] = 0;
        rc.qc->shadow = 0;
        rc.qc->hit = 0;
        rc.qc->extendWork = 0;
        rc.qc->shadowWork = 0;
    }
}

// i-th entry of queue pair `cur`: continuing paths first, then the ended ones
__device__ __forceinline__ uint32_t activeSlot(const RenderConst &rc, int cur, uint32_t i, uint32_t nCont)
{
    return i < nCont ? (cur ? rc.ps.contQ[1] : rc.ps.contQ[0])[i] : (cur ? rc.ps.regenQ[1] : rc.ps.regenQ[0])[i - nCont];
}

// miss.rmiss:16-39
__device__ __forceinline__ vec3 skyRadiance(const RenderConst &rc, vec3 dir)
{
    if ((rc.missFlags & PT_MISS_FLAGS_SKYBOX_2D) && rc.scene.hasSky2D)
    {
        const float longitude = atan2f(dir.z, dir.x);
        const float latitude = asinf(-dir.y);
        const float4 c = textureLod0(rc.scene, rc.scene.sky2D, longitude / 2.0f / PT_PI + 0.5f, latitude / PT_PI + 0.5f);
        const vec3 rgb = V3(c);
        return hdrToLdr(rgb);
    }
    if ((rc.missFlags & PT_MISS_FLAGS_SKYBOX_CUBE) && rc.scene.skyCubeSlot)
        return V3(sampleCube(rc.scene, rc.scene.skyCubeSlot, dir));
    return V3(0.08f, 0.09f, 0.1f);
}

// ---------------------------------------------------------------------------------------------
// extend
// ---------------------------------------------------------------------------------------------
// raygen.rgen:71-75, 99-117 and 38-58 for one ended path: finish its sample and start the slot's next
// one.  Called where k_extend would load the slot's ray, by a converged batch of regen-queue entries,
// so the lanes of a warp take consecutive work items (neighbouring pixels) with one atomic.
__device__ __forceinline__ RayPacket regeneratePath(const RenderConst &rc, uint32_t entry, uint32_t &samples, uint32_t &restarts)
{
    const uint32_t slot = entry & kSlotMask;
    const PathRecord &rec = rc.ps.rec[slot];
    const float4 rad4 = rec.rad, thr4 = rec.thr, d4 = rec.rayD;
    vec3 radiance = V3(rad4);
    if (entry & kRegenMiss) // miss.rmiss + raygen.rgen:71-75: the path ended with the sky radiance
        radiance = radiance + V3(thr4) * skyRadiance(rc, V3(d4));
    uint32_t item = __float_as_uint(rad4.w);
    const uint32_t state = __float_as_uint(thr4.w);
    const uint32_t restartCount = (state >> kRestartShift) & kRestartMask, smpl = state >> kSampleShift;
    const bool isBad = bad(radiance.x) || bad(radiance.y) || bad(radiance.z);
    // raygen.rgen:99-112: radiance = 0; smpl = -1 — ALL samples of the frame are redone with the ADVANCED rng state
    const bool restart = isBad && restartCount < kMaxRestarts;
    RayPacket p;
    p.slot = kDeadSlot;
    p.ox = p.oy = p.oz = p.dx = p.dy = p.dz = p.tmax = 0.0f;
    PrimaryRays pr;
    if (!restart)
        samples++; // one kept iteration of the sample loop (raygen.rgen:42) has ended
    if (restart || smpl + 1 < rc.samplesPerFrame)
    {
        const uint32_t s = item / rc.pixelCount, pi = item - s * rc.pixelCount;
        if (restart)
        {
            restarts++;
            pr = generatePath(rc, slot, __ldg(rc.pixelList + pi), item, __float_as_uint(d4.w), restartCount + 1);
        }
        else // the frame's next sample: same rng stream, radiance keeps summing (raygen.rgen:40-42)
            pr = generatePath(rc, slot, __ldg(rc.pixelList + pi), item, __float_as_uint(d4.w), restartCount, smpl + 1, radiance);
    }
    else
    {
        // park the frame's radiance; k_resolve adds the round's frames to the image in frame order
        rc.sbuf[item] = isBad ? make_float4(0.0f, 0.0f, 0.0f, 0.0f) : make_float4(radiance.x, radiance.y, radiance.z, 1.0f);
        item = atomicAggInc(rc.nextItem);
        if (item >= rc.itemCount)
            return p; // the round has no work left for this slot
        pr = startItem(rc, slot, item);
    }
    p.slot = slot;
    p.ox = pr.origin.x, p.oy = pr.origin.y, p.oz = pr.origin.z;
    p.dx = pr.direction.x, p.dy = pr.direction.y, p.dz = pr.direction.z;
    p.tmax = 10000.0f;
    return p;
}

template <bool ALPHA, bool STATS> __global__ void __launch_bounds__(128, PT_TRACE_MIN_BLOCKS) k_extend(RenderConst rc, int cur)
{
    const uint32_t nCont = rc.qc->cont[cur], n = nCont + rc.qc->regen[cur];
    // counters of k_shadow, which has completed (stream order) and is not running now
    if (blockIdx.x == 0 && threadIdx.x == 0)
    {
        rc.qc->shadow = 0;
        rc.qc->shadowWork = 0;
    }
    uint32_t hits = 0, rays = 0, samples = 0, restarts = 0;
    uint32_t *regenOut = cur ? rc.ps.regenQ[0] : rc.ps.regenQ[1];
    unsigned long long stack[PT_STACK_SIZE];
    Traverser<true, ALPHA, STATS> tr;
    tr.stack = stack;
    tr.st = TraversalStats { 0, 0, 0 };
    tracePersistent(
        rc.scene, n, &rc.qc->extendWork, tr, 0.00001f,
        [&](uint32_t i) { return activeSlot(rc, cur, i, nCont); },
        // force-inlined: as a call it forced a local-memory copy of the kernel parameter block (DESIGN.md §3)
        [&](uint32_t entry) __attribute__((always_inline)) {
            if (entry & kRegen)
                return regeneratePath(rc, entry, samples, restarts);
            RayPacket p;
            p.slot = entry;
            const float4 o = rc.ps.rec[p.slot].rayO, d = rc.ps.rec[p.slot].rayD;
            p.ox = o.x, p.oy = o.y, p.oz = o.z;
            p.dx = d.x, p.dy = d.y, p.dz = d.z;
            p.tmax = 10000.0f;
            return p;
        },
        [&](Traverser<true, ALPHA, STATS> &t, uint32_t slot) {
            rays++;
            if (t.hit.tri == 0xffffffffu)
            {
                // the path ends; its sample is finished by the next k_extend (regeneratePath)
                regenOut[atomicAggInc(&rc.qc->regen[cur ^ 1])] = slot | kRegen | kRegenMiss;
                return;
            }
            rc.ps.rec[slot].hit = make_float4(__uint_as_float(t.hit.tri), t.hit.t, t.hit.b1, t.hit.b2);
            if (ALPHA)
            {
                rc.ps.rec[slot].decal = make_float4(t.decal.r, t.decal.g, t.decal.b, t.decal.dist);
                rc.ps.rec[slot].decalA = t.decal.a;
            }
            const uint32_t pos = atomicAggInc(&rc.qc->hit);
            rc.ps.hitQ[pos] = slot;
            rc.ps.hitKey[pos] = t.hit.tri >> rc.hitKeyShift;
            hits++;
        },
        TailStats { rc.counters->visitHist, &rc.counters->warpIters, &rc.counters->warpDrainIters,
                    &rc.counters->maxWarpDrainIters });
    warpAdd(&rc.counters->hits, hits);
    warpAdd(&rc.counters->raysClosest, rays);
    warpAdd(&rc.counters->samples, samples);
    warpAdd(&rc.counters->restarts, restarts);
    if (STATS)
    {
        warpAdd(&rc.counters->boxClosest, tr.st.boxTests);
        warpAdd(&rc.counters->triClosest, tr.st.triTests);
        warpAdd(&rc.counters->alphaClosest, tr.st.alphaTests);
    }
}

// ---------------------------------------------------------------------------------------------
// material.glsl
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ MaterialSample sampleMaterial(const DeviceScene &s, uint32_t materialId, float u, float v,
                                                         float4 deriv, bool inside, bool flipNormalY, uint32_t *texels,
                                                         uint32_t debugFlags = 0)
{
    const uint32_t type = materialId & 0xffu, index = materialId >> 8;
    MaterialSample r;
    if (type > 2)
    {
        // material.glsl:163-166 leaves everything else undefined; zero like the oracle
        r = MaterialSample {};
        r.Color = V3(1.0f, 0.0f, 0.0f);
        r.EmissiveColor = V3(1.0f, 0.0f, 0.0f);
        return r;
    }
    const MaterialRaw *m = (type == 0 ? s.materials[0] : type == 1 ? s.materials[1] : s.materials[2]) + index;
    const float4 q0 = __ldg(&m->q[0]), q1 = __ldg(&m->q[1]), q2 = __ldg(&m->q[2]);
    const float4 q3 = __ldg(&m->q[3]), q4 = __ldg(&m->q[4]), q5 = __ldg(&m->q[5]);
    auto tex = [&](float idxBits) {
        const uint32_t slot = __float_as_uint(idxBits);
        if (texels)
            *texels += textureGradTexels(s, slot, deriv);
        return textureGrad(s, slot, u, v, deriv);
    };
    r.AttenuationColor = V3(q3.x, q3.y, q3.z);
    r.AttenuationDistance = q3.w;
    if (type == 0)
    {
        // material.glsl:62-84
        // (debug view only: sampleValue(flags, HitGroupFlagsDisable*Texture, ...), material.glsl:69-70)
        const float colorSlot = (debugFlags & PT_DEBUG_HIT_DISABLE_COLOR_TEXTURE) ? __uint_as_float(0u) : q5.x;
        const float normalSlot = (debugFlags & PT_DEBUG_HIT_DISABLE_NORMAL_TEXTURE) ? __uint_as_float(1u) : q5.y;
        const float4 e = tex(q4.w), c = tex(colorSlot), nm = tex(normalSlot);
        r.EmissiveColor = (V3(e) + V3(q0)) * q0.w;
        r.Color = V3(c) * V3(q1);
        r.Normal = reconstructNormalFromXY(nm);
        r.Roughness = tex(q5.z).y * q2.x;
        r.Metalness = tex(q5.w).z * q2.y;
        r.Transmission = q2.w;
        r.Eta = inside ? q2.z : (1.0f / q2.z);
    }
    else
    {
        // material.glsl:86-113 / 115-142 (specular-glossiness and Phong share the layout)
        const float colorSlot = (debugFlags & PT_DEBUG_HIT_DISABLE_COLOR_TEXTURE) ? __uint_as_float(0u) : q4.w;
        const float normalSlot = (debugFlags & PT_DEBUG_HIT_DISABLE_NORMAL_TEXTURE) ? __uint_as_float(1u) : q5.x;
        const float4 e = tex(q4.z), c = tex(colorSlot), nm = tex(normalSlot);
        r.EmissiveColor = (V3(e) + V3(q0)) * q0.w;
        r.Color = V3(c) * V3(q1);
        r.Normal = reconstructNormalFromXY(nm);
        r.Transmission = q4.y;
        r.Eta = inside ? q4.x : (1.0f / q4.x);
        const vec3 specular = V3(tex(q5.y)) * V3(q2);
        const float glossiness = tex(q5.z).w * q2.w;
        r.Roughness = 1.0f - glossiness;
        const vec3 diff = vmax(specular - 0.04f, 0.0f) / ((r.Color - 0.04f) + 0.00001f);
        r.Metalness = (diff.x + diff.y + diff.z) / 3.0f;
    }
    if (flipNormalY)
        r.Normal.y *= -1.0f;
    return r;
}

// ---------------------------------------------------------------------------------------------
// emissive-MIS light sampling (DESIGN.md §3g): a uniform point on emitter k of the table, seen from `position`.  Returns the
// light sample in sampleLight's form (Color = emission, Attenuation = 1 until the MIS weight is known) and its pdf in
// solid angle; pdf 0 when the point cannot be seen (grazing, or a degenerate triangle).
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ LightSample sampleEmitter(const DeviceScene &s, const EmitterTable &em, uint32_t k, float r1, float r2,
                                                     vec3 position, float &pdf)
{
    const float4 e0 = __ldg(em.rec + 4 * (size_t)k), e1 = __ldg(em.rec + 4 * (size_t)k + 1);
    const float4 e2 = __ldg(em.rec + 4 * (size_t)k + 2), e3 = __ldg(em.rec + 4 * (size_t)k + 3);
    const vec3 p0 = V3(e0.x, e0.y, e0.z), p1 = V3(e0.w, e1.x, e1.y), p2 = V3(e1.z, e1.w, e2.x);
    const float su = sqrtf(r1);
    const float b0 = 1.0f - su, b1 = su * (1.0f - r2), b2 = su * r2;
    const vec3 y = p0 * b0 + p1 * b1 + p2 * b2;
    const float u = e2.y * b0 + e2.w * b1 + e3.y * b2, v = e2.z * b0 + e3.x * b1 + e3.z * b2;
    const vec3 ng = normalize(cross(p1 - p0, p2 - p0));
    // the shadow ray's target leaves the emitter towards the shading point, so the emitter cannot occlude itself
    const vec3 target = offsetRayOriginSelfIntersection(y, dot(ng, position - y) >= 0.0f ? ng : -ng);
    LightSample r;
    r.Distance = length(position - target);
    r.Direction = normalize(position - target);
    float4 q0;
    uint32_t slot;
    emissiveSource(s, __float_as_uint(e3.w), q0, slot);
    r.Color = (V3(textureLod0(s, s.textures[slot], u, v)) + V3(q0)) * q0.w;
    r.Attenuation = 1.0f;
    const float cosLight = fabsf(dot(ng, r.Direction));
    pdf = em.pEmitter * __ldg(em.emitterPdf + k) * (r.Distance * r.Distance) / cosLight;
    if (!(pdf > 0.0f) || isinf(pdf))
        pdf = 0.0f;
    return r;
}

// ---------------------------------------------------------------------------------------------
// shade: closestHit.rchit, then the raygen bounce logic (misses are finished by k_extend).
// EMISSIVE adds emissive-triangle light sampling and MIS (pt_set_light_sampling, DESIGN.md §3g) to the same closest-hit
// and bounce logic and the same main rng stream: the emitter branch of the light sample, the MIS weight of emission found
// by BSDF sampling and the previous bounce's BSDF pdf in the path record; em is read only when EMISSIVE.  The body stays
// in the kernel: moving it into a force-inlined __device__ function changed the machine code of both modes.
// ---------------------------------------------------------------------------------------------
template <bool ALPHA, bool STATS, bool EMISSIVE>
__global__ void __launch_bounds__(128, PT_SHADE_MIN_BLOCKS) k_shade(RenderConst rc, int cur, EmitterTable em)
{
    const uint32_t n = rc.qc->hit;
    const uint32_t stride = gridDim.x * blockDim.x;
    const DeviceScene &s = rc.scene;
    uint32_t texels = 0;
    // the queue positions of k_extend, which has completed (stream order)
    if (blockIdx.x == 0 && threadIdx.x == 0)
        rc.qc->extendWork = 0;
    const uint32_t *hitQueue = rc.sortHits ? rc.ps.hitQSorted : rc.ps.hitQ;
    // (requesting the next hit's path record into L2 one loop iteration ahead was measured: no gain,
    // the kernel is bound by issue latency at 16 warps per SM, not by the record's DRAM latency)
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
    {
        const uint32_t slot = hitQueue[i];
        const float4 hitv = rc.ps.rec[slot].hit;
        const float4 rayO = rc.ps.rec[slot].rayO, rayD = rc.ps.rec[slot].rayD;
        // read with the rest of the record: reading throughput, radiance and the differentials again where they are
        // used exposed the loads' latency at the end of every hit (measured: k_shade +12 %, chess)
        float4 thr4 = rc.ps.rec[slot].thr;
        float4 rad4 = rc.ps.rec[slot].rad;
        vec3 throughput = V3(thr4), radiance = V3(rad4);
        uint32_t state = __float_as_uint(thr4.w);
        const vec3 rayDir = V3(rayD);
        const uint32_t tri = __float_as_uint(hitv.x);

        uint32_t rng = __float_as_uint(rayD.w);
        float maxRoughness = rayO.w;
        const float rayTmax = hitv.y;
        const vec3 bary = V3(1.0f - hitv.z - hitv.w, hitv.z, hitv.w);

        // ---- closestHit.rchit:54-83 with baked world-space data ---------------------------------
        const float4 q0 = __ldg(s.triPos + 3 * (size_t)tri), q1 = __ldg(s.triPos + 3 * (size_t)tri + 1);
        const float4 q2 = __ldg(s.triPos + 3 * (size_t)tri + 2);
        const TriShade &ts = s.triShade[__float_as_uint(q0.w)];
        const float4 a0 = __ldg(&ts.a[0]), a1 = __ldg(&ts.a[1]), a2 = __ldg(&ts.a[2]), a3 = __ldg(&ts.a[3]);
        const float4 a4 = __ldg(&ts.a[4]), a5 = __ldg(&ts.a[5]), a6 = __ldg(&ts.a[6]), a7 = __ldg(&ts.a[7]);
        const float4 a8 = __ldg(&ts.a[8]);
        const uint32_t materialId = __float_as_uint(q2.w);
        const vec3 p0 = V3(q0), p1 = V3(q1), p2 = V3(q2);
        const vec3 n0r = V3(a0.x, a0.y, a0.z), n1r = V3(a0.w, a1.x, a1.y), n2r = V3(a1.z, a1.w, a2.x);
        const vec3 t0r = V3(a2.y, a2.z, a2.w), t1r = V3(a3.x, a3.y, a3.z), t2r = V3(a3.w, a4.x, a4.y);
        const vec3 b0r = V3(a4.z, a4.w, a5.x), b1r = V3(a5.y, a5.z, a5.w), b2r = V3(a6.x, a6.y, a6.z);
        const vec2 uv0 = V2(a6.w, a7.x), uv1 = V2(a7.y, a7.z), uv2 = V2(a7.w, a8.x);
        // MIS weight of the emission this BSDF-sampled ray found (bounce >= 1 on a triangle the light sampling can pick)
        float emissionWeight = 1.0f;
        if (EMISSIVE && (state & 0xffu) != 0)
        {
            const float pdfOverArea = __ldg(em.pdfOverArea + __float_as_uint(q0.w));
            if (pdfOverArea > 0.0f)
            {
                const float4 a11 = __ldg(&ts.a[11]);
                const float cosLight = fabsf(a11.y * rayDir.x + a11.z * rayDir.y + a11.w * rayDir.z);
                const float pdfLight = em.pEmitter * pdfOverArea * (rayTmax * rayTmax) / cosLight;
                emissionWeight = powerHeuristic(__uint_as_float(rc.ps.rec[slot].pad[0]), pdfLight);
            }
        }

        const vec3 position = p0 * bary.x + p1 * bary.y + p2 * bary.z;
        const vec2 texCoords = uv0 * bary.x + uv1 * bary.y + uv2 * bary.z;
        vec3 normal = normalize(n0r * bary.x + n1r * bary.y + n2r * bary.z);
        vec3 tangent = normalize(t0r * bary.x + t1r * bary.y + t2r * bary.z);
        vec3 bitangent = normalize(b0r * bary.x + b1r * bary.y + b2r * bary.z);
        const vec3 edge1 = p1 - p0, edge2 = p2 - p0;
        // normalised once per triangle by k_bake (same functions, same operands)
        const float4 a9 = __ldg(&ts.a[9]), a10 = __ldg(&ts.a[10]), a11 = __ldg(&ts.a[11]);
        const vec3 n0 = V3(a9.x, a9.y, a9.z), n1 = V3(a9.w, a10.x, a10.y), n2 = V3(a10.z, a10.w, a11.x);
        vec3 geometricNormal = V3(a11.y, a11.z, a11.w);
        const bool inside = dot(geometricNormal, rayDir) > 0.0f;
        if (inside)
        {
            geometricNormal = -geometricNormal;
            normal = -normal;
            tangent = -tangent;
            bitangent = -bitangent;
        }

        // ---- tracing.glsl:2-28 -------------------------------------------------------------
        vec3 dpdu, dpdv, dndu, dndv;
        computeDpnDuv(edge1, edge2, n1 - n0, n2 - n0, uv1 - uv0, uv2 - uv0, tangent, bitangent, dpdu, dpdv, dndu, dndv);
        const float4 d0 = rc.ps.rec[slot].diff0, d1 = rc.ps.rec[slot].diff1, d2 = rc.ps.rec[slot].diff2;
        RayDifferentials rd;
        rd.rxOrigin = V3(d0.x, d0.y, d0.z);
        rd.rxDirection = V3(d0.w, d1.x, d1.y);
        rd.ryOrigin = V3(d1.z, d1.w, d2.x);
        rd.ryDirection = V3(d2.y, d2.z, d2.w);
        vec3 dpdx, dpdy;
        computeDpDxy(position, rd.rxOrigin, rd.rxDirection, rd.ryOrigin, rd.ryDirection, normal, dpdx, dpdy);
        const float4 derivatives = computeDerivatives(dpdx, dpdy, dpdu, dpdv);
        // Register diet: what the code AFTER the BSDF sample needs of the geometry is reduced to its results now — the
        // ray origin of either outcome (reflected / refracted: same operations as the one call the shader makes, for
        // both values of its flag) and the normal's screen-space derivatives — so that the triangle's corners, vertex
        // normals, barycentrics and uv derivatives are dead while the material and the BSDF are evaluated.
        const vec3 originReflected = offsetRayOriginShadowTerminator(position, p0, p1, p2, n0, n1, n2, bary, false);
        const vec3 originRefracted = offsetRayOriginShadowTerminator(position, p0, p1, p2, n0, n1, n2, bary, true);
        const vec3 originThrough = offsetRayOriginSelfIntersection(position, -geometricNormal);
        const vec3 dndx = dndu * derivatives.x + dndv * derivatives.y;
        const vec3 dndy = dndu * derivatives.z + dndv * derivatives.w;

        // ---- material, closestHit.rchit:101-117 -------------------------------------------------
        MaterialSample material = sampleMaterial(s, materialId, texCoords.x, texCoords.y, derivatives, inside,
                                                 (rc.hitFlags & PT_HIT_FLAGS_DX_NORMAL_TEXTURES) != 0,
                                                 STATS ? &texels : nullptr);
        if (ALPHA)
        {
            const float4 dec = rc.ps.rec[slot].decal;
            if (dec.w != -1.0f && rayTmax > dec.w)
                material.Color = mix(material.Color, V3(dec), rc.ps.rec[slot].decalA);
        }
        maxRoughness = fmaxf(material.Roughness, maxRoughness);
        material.Roughness = fmaxf(maxRoughness, 0.01f);

        const mat3 geometryTBN = mat3 { tangent, bitangent, normal };
        const vec3 N = normalize(normal + mul(geometryTBN, material.Normal));
        const mat3 TBN = computeTangentSpace(N);
        // TBN is orthonormal: inverse(TBN) == transpose(TBN)
        const vec3 V = normalize(mulT(TBN, normalize(-rayDir)));

        BSDFSample bsdf = sampleBSDF(material, V, rng);

        if (inside)
        {
            const float e = rayTmax / material.AttenuationDistance;
            bsdf.Color.x *= powf(material.AttenuationColor.x, e);
            bsdf.Color.y *= powf(material.AttenuationColor.y, e);
            bsdf.Color.z *= powf(material.AttenuationColor.z, e);
        }
        const bool isRefracted = bsdf.Direction.z < 0.0f;
        const vec3 rayOrigin = isRefracted ? originRefracted : originReflected;

        float lightPdf, lightSmplPdf;
        const float l0 = rnd(rng);
        const float l1 = rnd(rng);
        const float l2 = rnd(rng);
        LightSample light = sampleLight(s.lights, V3(l0, l1, l2), rayOrigin, lightPdf);
        bool emitterSample = false;
        if (EMISSIVE)
        {
            // the branch, the alias draw (bucket, 32-bit fraction) and the point come from a secondary stream
            uint32_t rng2 = lightSampleRng(rng);
            if (rnd(rng2) < em.pEmitter)
            {
                const uint32_t hi = xorshift(rng2), lo = xorshift(rng2);
                const uint32_t bucket = __umulhi(hi, em.count);
                const uint2 entry = __ldg(em.alias + bucket);
                const uint32_t k = lo < entry.x ? bucket : entry.y;
                const float r1 = rnd(rng2);
                const float r2 = rnd(rng2);
                light = sampleEmitter(s, em, k, r1, r2, rayOrigin, lightPdf);
                emitterSample = true;
                // the last bounce: the reference mode never collects emission one vertex further, so neither does this
                if ((state & 0xffu) + 1 >= rc.bounceCount)
                    lightPdf = 0.0f;
            }
            else
                lightPdf = lightPdf * (1.0f - em.pEmitter);
        }
        const vec3 L = normalize(mulT(TBN, -light.Direction));
        const vec3 lightBsdf = evaluateBSDF(material, V, L, lightSmplPdf);
        if (EMISSIVE && emitterSample)
            light.Attenuation = powerHeuristic(lightPdf, lightSmplPdf);

        const vec3 newDir = normalize(mul(TBN, bsdf.Direction));
        const vec3 newPos = isRefracted ? originThrough : rayOrigin;
        const vec3 directLight = light.Color * light.Attenuation * lightBsdf;

        propagateDifferentials(normal, rayOrigin, -rayDir, newDir, dndx, dndy, material.Eta, isRefracted, rd);

        // ---- raygen.rgen:71-96 ----------------------------------------------------------------
        radiance += throughput * (EMISSIVE ? material.EmissiveColor * emissionWeight : material.EmissiveColor);
        bool done = false;
        if (bsdf.Pdf == -1.0f)
            done = true; // raygen.rgen:71 cannot tell this from a miss
        else
        {
            if (lightPdf > 0.0f)
            {
                const vec3 c = throughput * directLight / lightPdf;
                // a contribution of exactly +-0 cannot change the radiance: the occlusion query is skipped.  A non-finite
                // emitter sample is dropped: it must not cause a NaN/Inf restart the reference mode would not make.
                if (!(c.x == 0.0f && c.y == 0.0f && c.z == 0.0f) &&
                    !(EMISSIVE && emitterSample && (bad(c.x) || bad(c.y) || bad(c.z))))
                {
                    const vec3 sd = -normalize(light.Direction);
                    rc.ps.rec[slot].shO = make_float4(newPos.x, newPos.y, newPos.z, light.Distance);
                    rc.ps.rec[slot].shD = make_float4(sd.x, sd.y, sd.z, 0.0f);
                    rc.ps.rec[slot].shC = make_float4(c.x, c.y, c.z, 0.0f);
                    rc.ps.shadowQueue[atomicAggInc(&rc.qc->shadow)] = slot;
                }
            }
            if (bsdf.Pdf > 0.001f)
                throughput *= bsdf.Color / bsdf.Pdf;
            const float prob = fminf(maxComponent(throughput), 1.0f);
            if (prob < 0.001f)
                done = true;
            else if (prob < rnd(rng))
                done = true;
            else
                throughput = throughput / prob;
        }
        const uint32_t bounce = (state & 0xffu) + 1;
        if (bounce >= rc.bounceCount)
            done = true;
        state = (state & ~0xffu) | bounce;
        // continuing paths go straight to the next iteration's queue (in shading = triangle order, so
        // the next extend starts from spatially coherent origins); ended ones to its regen queue
        // (their shadow ray, if any, is resolved by k_shadow before that)
        if (done)
            (cur ? rc.ps.regenQ[0] : rc.ps.regenQ[1])[atomicAggInc(&rc.qc->regen[cur ^ 1])] = slot | kRegen;
        else
            (cur ? rc.ps.contQ[0] : rc.ps.contQ[1])[atomicAggInc(&rc.qc->cont[cur ^ 1])] = slot;

        rc.ps.rec[slot].rad = make_float4(radiance.x, radiance.y, radiance.z, rad4.w);
        // the rng state outlives the path (a NaN/Inf restart continues the stream, raygen.rgen:99-112)
        rc.ps.rec[slot].rayD = make_float4(newDir.x, newDir.y, newDir.z, __uint_as_float(rng));
        if (!done)
        {
            rc.ps.rec[slot].thr = make_float4(throughput.x, throughput.y, throughput.z, __uint_as_float(state));
            rc.ps.rec[slot].rayO = make_float4(newPos.x, newPos.y, newPos.z, maxRoughness);
            rc.ps.rec[slot].diff0 = make_float4(rd.rxOrigin.x, rd.rxOrigin.y, rd.rxOrigin.z, rd.rxDirection.x);
            rc.ps.rec[slot].diff1 = make_float4(rd.rxDirection.y, rd.rxDirection.z, rd.ryOrigin.x, rd.ryOrigin.y);
            rc.ps.rec[slot].diff2 = make_float4(rd.ryOrigin.z, rd.ryDirection.x, rd.ryDirection.y, rd.ryDirection.z);
            if (EMISSIVE)
                rc.ps.rec[slot].pad[0] = __float_as_uint(bsdf.Pdf);
        }
    }
    if (STATS)
        warpAdd(&rc.counters->texels, texels);
}

// ---------------------------------------------------------------------------------------------
// shadow
// ---------------------------------------------------------------------------------------------
template <bool ALPHA, bool STATS> __global__ void __launch_bounds__(128, PT_TRACE_MIN_BLOCKS) k_shadow(RenderConst rc, int cur)
{
    const uint32_t n = rc.qc->shadow;
    // Counters of the queues the NEXT iteration fills: this iteration's inputs.  Nothing in this
    // kernel reads them, and everything that did has completed (stream order).
    if (blockIdx.x == 0 && threadIdx.x == 0)
    {
        rc.qc->cont[cur] = 0;
        rc.qc->regen[cur] = 0;
        rc.qc->hit = 0;
    }
    unsigned long long stack[PT_STACK_SIZE];
    Traverser<false, ALPHA, STATS> tr;
    tr.stack = stack;
    tr.st = TraversalStats { 0, 0, 0 };
    tracePersistent(
        rc.scene, n, &rc.qc->shadowWork, tr, 0.00001f,
        [&](uint32_t i) { return rc.ps.shadowQueue[i]; },
        [&](uint32_t slot) {
            RayPacket p;
            p.slot = slot;
            const float4 o = rc.ps.rec[p.slot].shO, d = rc.ps.rec[p.slot].shD;
            p.ox = o.x, p.oy = o.y, p.oz = o.z;
            p.dx = d.x, p.dy = d.y, p.dz = d.z;
            p.tmax = o.w;
            return p;
        },
        [&](Traverser<false, ALPHA, STATS> &t, uint32_t slot) {
            if (t.hit.tri == 0xffffffffu)
            {
                const float4 c = rc.ps.rec[slot].shC;
                float4 r = rc.ps.rec[slot].rad;
                r.x += c.x;
                r.y += c.y;
                r.z += c.z;
                rc.ps.rec[slot].rad = r;
            }
        },
        TailStats { rc.counters->visitHist, &rc.counters->warpIters, &rc.counters->warpDrainIters,
                    &rc.counters->maxWarpDrainIters });
    if (STATS)
    {
        warpAdd(&rc.counters->boxShadow, tr.st.boxTests);
        warpAdd(&rc.counters->triShadow, tr.st.triTests);
        warpAdd(&rc.counters->alphaShadow, tr.st.alphaTests);
    }
    if (blockIdx.x == 0 && threadIdx.x == 0)
        atomicAdd(&rc.counters->raysShadow, (unsigned long long)n);
}

// ---------------------------------------------------------------------------------------------
// resolve: acc += radiance, one sample after the other (raygen.rgen:115-117 over consecutive frames)
// ---------------------------------------------------------------------------------------------
// ADAPTIVE adds the Welford update of the pixel's luminance statistics per sample (DESIGN.md §3i); a dropped frame
// (parked as 0) is a sample of luminance 0, as in the accumulation.  state is read only when ADAPTIVE.
template <bool ADAPTIVE> __global__ void __launch_bounds__(256) k_resolve(RenderConst rc, AdaptivePixel *state)
{
    const uint32_t stride = gridDim.x * blockDim.x;
    for (uint32_t pi = blockIdx.x * blockDim.x + threadIdx.x; pi < rc.pixelCount; pi += stride)
    {
        const uint32_t pixel = __ldg(rc.pixelList + pi);
        float4 a = rc.accum[pixel];
        AdaptivePixel st = ADAPTIVE ? state[pixel] : AdaptivePixel {};
        for (uint32_t s = 0; s < rc.roundSamples; s++)
        {
            const float4 r = __ldcs(rc.sbuf + (size_t)s * rc.pixelCount + pi);
            a.x = r.x + a.x;
            a.y = r.y + a.y;
            a.z = r.z + a.z;
            if (ADAPTIVE)
            {
                const float l = (0.2126f * r.x + 0.7152f * r.y) + 0.0722f * r.z;
                st.count += 1;
                const float d = l - st.mean;
                st.mean += d / (float)st.count;
                st.m2 += d * (l - st.mean);
            }
        }
        a.w = 1.0f;
        rc.accum[pixel] = a;
        if (ADAPTIVE)
            state[pixel] = st;
    }
}

// ---------------------------------------------------------------------------------------------
// standalone queries
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ pt_hit toPtHit(const DeviceScene &s, const Hit &h)
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

template <bool ALPHA> __global__ void k_first_hit(DeviceScene s, CameraMatrices cam, uint32_t width, uint32_t height, pt_hit *out)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= width * height)
        return;
    const uint32_t px = i % width, py = i / width;
    // ray.glsl:87-90: pixel centre
    const PrimaryRays pr = constructPrimaryRay((float)px, (float)py, (float)width, (float)height, cam, V2(0.5f, 0.5f),
                                               V2(0.0f, 0.0f), 0.0f, 0.0f);
    Hit hit;
    Decal decal;
    TraversalStats st;
    traverse<true, ALPHA, false>(s, pr.origin, pr.direction, 0.00001f, 10000.0f, hit, decal, st);
    out[i] = toPtHit(s, hit);
}

// ---------------------------------------------------------------------------------------------
// The reference's debug pipeline (Debug/debugRaygen.rgen, debugClosestHit.rchit, debugAnyhit.rahit,
// debugMiss.rmiss): one pixel-centre ray per pixel, a view of the first hit.  A diagnostics path,
// one thread per pixel with the plain per-thread traversal.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ vec3 debugRandomColor(uint32_t x) // debugClosestHit.rchit:141-161
{
    x *= 0x1eca7d79u;
    x ^= x >> 20;
    x = (x << 8) | (x >> 24);
    x = ~x;
    x ^= x << 5;
    x += 0x10afe4e7u;
    return V3((float)((x & 0xff000000u) >> 24) / 255.0f, (float)((x & 0x00ff0000u) >> 16) / 255.0f,
              (float)((x & 0x0000ff00u) >> 8) / 255.0f);
}

// debugClosestHit.rchit:70-139
__device__ __forceinline__ vec3 debugLightContribution(vec3 lightDir, vec3 lightColor, float attenuation, vec3 V, vec3 N, vec3 color,
                                                       float roughness, float metalness)
{
    const vec3 L = -normalize(lightDir);
    const vec3 H = normalize(V + L);
    const vec3 radiance = lightColor * attenuation;
    const vec3 F0 = mix(V3(0.04f), color, metalness);
    const float a = roughness * roughness, a2 = a * a;
    const float NdotH = fmaxf(dot(N, H), 0.0f), NdotH2 = NdotH * NdotH;
    float denomD = NdotH2 * (a2 - 1.0f) + 1.0f;
    denomD = PT_PI * denomD * denomD;
    const float NDF = a2 / fmaxf(denomD, 0.0001f);
    const float NdotV = fmaxf(dot(N, V), 0.0f), NdotL = fmaxf(dot(N, L), 0.0f);
    const float rr = roughness + 1.0f, k = (rr * rr) / 8.0f;
    const float ggx2 = NdotV / (NdotV * (1.0f - k) + k), ggx1 = NdotL / (NdotL * (1.0f - k) + k);
    const float G = ggx1 * ggx2;
    const float cosTheta = fmaxf(dot(H, V), 0.0f);
    const vec3 F = F0 + (V3(1.0f) - F0) * powf(clampf(1.0f - cosTheta, 0.0f, 1.0f), 5.0f);
    const vec3 numerator = F * (NDF * G);
    const float denominator = 4.0f * fmaxf(dot(N, V), 0.0f) * fmaxf(dot(N, L), 0.0f);
    const vec3 specular = numerator / fmaxf(denominator, 0.0001f);
    vec3 kD = V3(1.0f) - F;
    kD = kD * (1.0f - metalness);
    return (kD * color / PT_PI + specular) * radiance * NdotL;
}

// The pixel-centre primary hit of k_debug and k_denoise_guides (debugRaygen.rgen + debugClosestHit.rchit:163-265 on the
// baked world-space triangle): the surface, its material (textureGrad with the ray-differential derivatives, the decal mixed
// into the base colour on alpha scenes) and the normal-mapped shading normal N.  flags are PT_DEBUG_HIT_* bits.
struct PrimarySurface
{
    PrimaryRays pr;
    Hit hit;
    vec3 bary, p0, p1, p2, n0r, n1r, n2r, position, normal, N;
    vec2 texCoords;
    float4 ids; // TriShade a[8]: -, instance, geometry, primitive (bits)
    float4 derivatives;
    MaterialSample material;
};

// false on a miss (sf.pr and sf.hit are set)
template <bool ALPHA_PRIMARY, bool CULL>
__device__ __forceinline__ bool tracePrimarySurface(const DeviceScene &s, const CameraMatrices &cam, uint32_t px, uint32_t py,
                                                    uint32_t width, uint32_t height, uint32_t flags, PrimarySurface &sf)
{
    sf.pr = constructPrimaryRay((float)px, (float)py, (float)width, (float)height, cam, V2(0.5f, 0.5f), V2(0.0f, 0.0f), 0.0f, 0.0f);
    const PrimaryRays &pr = sf.pr;
    Hit &hit = sf.hit;
    Decal decal;
    TraversalStats st;
    traverse<true, ALPHA_PRIMARY, false, CULL>(s, pr.origin, pr.direction, 0.00001f, 10000.0f, hit, decal, st);
    if (hit.tri == 0xffffffffu)
        return false;

    const uint32_t tri = hit.tri;
    const vec3 bary = V3(1.0f - hit.b1 - hit.b2, hit.b1, hit.b2);
    const float4 q0 = __ldg(s.triPos + 3 * (size_t)tri), q1 = __ldg(s.triPos + 3 * (size_t)tri + 1);
    const float4 q2 = __ldg(s.triPos + 3 * (size_t)tri + 2);
    const TriShade &ts = s.triShade[__float_as_uint(q0.w)];
    const float4 a0 = __ldg(&ts.a[0]), a1 = __ldg(&ts.a[1]), a2 = __ldg(&ts.a[2]), a3 = __ldg(&ts.a[3]);
    const float4 a4 = __ldg(&ts.a[4]), a5 = __ldg(&ts.a[5]), a6 = __ldg(&ts.a[6]), a7 = __ldg(&ts.a[7]);
    const float4 a8 = __ldg(&ts.a[8]);
    const uint32_t materialId = __float_as_uint(q2.w);
    const vec3 p0 = V3(q0), p1 = V3(q1), p2 = V3(q2);
    const vec3 n0r = V3(a0.x, a0.y, a0.z), n1r = V3(a0.w, a1.x, a1.y), n2r = V3(a1.z, a1.w, a2.x);
    const vec3 t0r = V3(a2.y, a2.z, a2.w), t1r = V3(a3.x, a3.y, a3.z), t2r = V3(a3.w, a4.x, a4.y);
    const vec3 b0r = V3(a4.z, a4.w, a5.x), b1r = V3(a5.y, a5.z, a5.w), b2r = V3(a6.x, a6.y, a6.z);
    const vec2 uv0 = V2(a6.w, a7.x), uv1 = V2(a7.y, a7.z), uv2 = V2(a7.w, a8.x);
    const vec3 position = p0 * bary.x + p1 * bary.y + p2 * bary.z;
    const vec2 texCoords = uv0 * bary.x + uv1 * bary.y + uv2 * bary.z;
    const vec3 normal = normalize(n0r * bary.x + n1r * bary.y + n2r * bary.z);
    const vec3 tangent = normalize(t0r * bary.x + t1r * bary.y + t2r * bary.z);
    const vec3 bitangent = normalize(b0r * bary.x + b1r * bary.y + b2r * bary.z);

    // tracing.glsl:2-28
    vec3 dpdu, dpdv;
    {
        const vec3 edge1 = p1 - p0, edge2 = p2 - p0;
        const vec2 duv1 = uv1 - uv0, duv2 = uv2 - uv0;
        const float det = duv1.x * duv2.y - duv2.x * duv1.y;
        if (fabsf(det) < 1e-8f)
        {
            dpdu = tangent;
            dpdv = bitangent;
        }
        else
        {
            const float invDet = 1.0f / det;
            dpdu = (duv2.y * edge1 - duv1.y * edge2) * invDet;
            dpdv = (-duv2.x * edge1 + duv1.x * edge2) * invDet;
        }
    }
    // tracing.glsl:31-41 with both offset rays starting at the camera
    vec3 dpdx, dpdy;
    {
        const float d = -dot(normal, position);
        const float tx = (-dot(normal, pr.origin) - d) / dot(normal, pr.rxDirection);
        const float ty = (-dot(normal, pr.origin) - d) / dot(normal, pr.ryDirection);
        dpdx = (pr.origin + tx * pr.rxDirection) - position;
        dpdy = (pr.origin + ty * pr.ryDirection) - position;
    }
    const float4 derivatives =
        (flags & PT_DEBUG_HIT_DISABLE_MIP_MAPS) ? make_float4(0.0f, 0.0f, 0.0f, 0.0f) : computeDerivatives(dpdx, dpdy, dpdu, dpdv);
    MaterialSample material = sampleMaterial(s, materialId, texCoords.x, texCoords.y, derivatives, false,
                                             (flags & PT_DEBUG_HIT_DX_NORMAL_TEXTURES) != 0, nullptr, flags);
    if (ALPHA_PRIMARY && decal.dist != -1.0f && hit.t > decal.dist)
        material.Color = mix(material.Color, V3(decal.r, decal.g, decal.b), decal.a);
    const mat3 TBN = mat3 { tangent, bitangent, normal };
    sf.N = normalize(normal + mul(TBN, material.Normal));
    sf.bary = bary;
    sf.p0 = p0;
    sf.p1 = p1;
    sf.p2 = p2;
    sf.n0r = n0r;
    sf.n1r = n1r;
    sf.n2r = n2r;
    sf.position = position;
    sf.normal = normal;
    sf.texCoords = texCoords;
    sf.ids = a8;
    sf.derivatives = derivatives;
    sf.material = material;
    return true;
}

template <bool ALPHA_PRIMARY, bool ALPHA_SHADOW, bool CULL>
__global__ void k_debug(DeviceScene s, CameraMatrices cam, uint32_t width, uint32_t height, uint32_t missFlags, pt_debug_params dbg,
                        float4 *out)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= width * height)
        return;
    const uint32_t px = i % width, py = i / width;
    const uint32_t flags = dbg.hit_group_flags;
    PrimarySurface sf;
    if (!tracePrimarySurface<ALPHA_PRIMARY, CULL>(s, cam, px, py, width, height, flags, sf))
    {
        // debugMiss.rmiss:17-36 (no hdrToLdr here)
        const PrimaryRays &pr = sf.pr;
        vec3 c = V3(0.2f, 0.2f, 0.2f);
        if ((missFlags & PT_MISS_FLAGS_SKYBOX_2D) && s.hasSky2D)
        {
            const float longitude = atan2f(pr.direction.z, pr.direction.x), latitude = asinf(-pr.direction.y);
            c = V3(textureLod0(s, s.sky2D, longitude / 2.0f / PT_PI + 0.5f, latitude / PT_PI + 0.5f));
        }
        else if ((missFlags & PT_MISS_FLAGS_SKYBOX_CUBE) && s.skyCubeSlot)
            c = V3(sampleCube(s, s.skyCubeSlot, pr.direction));
        out[i] = make_float4(c.x, c.y, c.z, 1.0f);
        return;
    }
    const vec3 bary = sf.bary, p0 = sf.p0, p1 = sf.p1, p2 = sf.p2, position = sf.position, N = sf.N;
    const vec3 n0 = normalize(sf.n0r), n1 = normalize(sf.n1r), n2 = normalize(sf.n2r);
    const vec2 texCoords = sf.texCoords;
    const float4 derivatives = sf.derivatives, a8 = sf.ids;
    const MaterialSample &material = sf.material;
    const vec3 V = -normalize(sf.pr.direction);

    vec3 result;
    switch (dbg.render_mode)
    {
    case PT_DEBUG_MODE_WORLD_POSITION: result = position; break;
    case PT_DEBUG_MODE_NORMAL: result = N; break;
    case PT_DEBUG_MODE_TEXTURE_COORDS: result = V3(texCoords.x, texCoords.y, 0.0f); break;
    case PT_DEBUG_MODE_MIPS: {
        // tracing.glsl:151-161
        const float sx = sqrtf(derivatives.x * derivatives.x + derivatives.y * derivatives.y);
        const float sy = sqrtf(derivatives.z * derivatives.z + derivatives.w * derivatives.w);
        const float smax = fmaxf(sx, sy);
        result = V3(0.1f * (smax == 0.0f ? 0.0f : log2f(smax)) + 1.0f);
        break;
    }
    case PT_DEBUG_MODE_GEOMETRY: result = debugRandomColor(__float_as_uint(a8.z)); break;
    case PT_DEBUG_MODE_PRIMITIVE: result = debugRandomColor(__float_as_uint(a8.w)); break;
    case PT_DEBUG_MODE_INSTANCE: result = debugRandomColor(__float_as_uint(a8.y)); break;
    default: {
        const float ambient = 0.1f;
        vec3 totalLight = material.Color * ambient + material.EmissiveColor;
        vec3 tmpu = position - p0, tmpv = position - p1, tmpw = position - p2;
        const float dotu = fminf(0.0f, dot(tmpu, n0)), dotv = fminf(0.0f, dot(tmpv, n1)), dotw = fminf(0.0f, dot(tmpw, n2));
        tmpu = tmpu - n0 * dotu;
        tmpv = tmpv - n1 * dotv;
        tmpw = tmpw - n2 * dotw;
        const vec3 Pp = position + tmpu * bary.x + tmpv * bary.y + tmpw * bary.z;
        const bool shadowsDisabled = (flags & PT_DEBUG_HIT_DISABLE_SHADOWS) != 0;
        auto occluded = [&](vec3 lightDir, float dist) {
            Hit h;
            Decal dd;
            TraversalStats st2;
            traverse<false, ALPHA_SHADOW, false>(s, Pp, -normalize(lightDir), 0.00001f, dist, h, dd, st2);
            return h.tri != 0xffffffffu;
        };
        const LightBlock *lb = s.lights;
        const vec3 dirDirection = V3(__ldg(&lb->dirDirection)), dirColor = V3(__ldg(&lb->dirColor));
        if (shadowsDisabled || !occluded(dirDirection, 100000.0f))
            totalLight = totalLight + debugLightContribution(dirDirection, dirColor, 1.0f, V, N, material.Color, material.Roughness,
                                                             material.Metalness);
        const uint32_t count = __ldg(&lb->count);
        for (uint32_t li = 0; li < count; li++)
        {
            const float4 lc = __ldg(&lb->point[li * 3]), lp = __ldg(&lb->point[li * 3 + 1]), la = __ldg(&lb->point[li * 3 + 2]);
            const vec3 lightDirection = Pp - V3(lp);
            const float dist = length(lightDirection);
            const float attenuation = 1.0f / (la.x + dist * la.y + dist * dist * la.z);
            if (shadowsDisabled || !occluded(lightDirection, dist))
                totalLight = totalLight + debugLightContribution(lightDirection, V3(lc), attenuation, V, N, material.Color,
                                                                 material.Roughness, material.Metalness);
        }
        result = totalLight;
    }
    }
    out[i] = make_float4(result.x, result.y, result.z, 1.0f);
}

// Guides of the denoiser (denoise.cu): k_debug's primary surface with its default flags, per pixel (base colour, hit
// distance t; t = -1 on a miss) and (shading normal N, 0)
template <bool ALPHA>
__global__ void k_denoise_guides(DeviceScene s, CameraMatrices cam, uint32_t width, uint32_t height, uint32_t flags, float4 *albedoT,
                                 float4 *normal)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= width * height)
        return;
    PrimarySurface sf;
    if (!tracePrimarySurface<ALPHA, false>(s, cam, i % width, i / width, width, height, flags, sf))
    {
        albedoT[i] = make_float4(0.0f, 0.0f, 0.0f, -1.0f);
        normal[i] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        return;
    }
    const vec3 c = sf.material.Color;
    albedoT[i] = make_float4(c.x, c.y, c.z, sf.hit.t);
    normal[i] = make_float4(sf.N.x, sf.N.y, sf.N.z, 0.0f);
}

template <bool ALPHA> __global__ void k_trace_closest(DeviceScene s, const pt_ray *rays, uint64_t n, pt_hit *out)
{
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n)
        return;
    const pt_ray r = rays[i];
    Hit hit;
    Decal decal;
    TraversalStats st;
    traverse<true, ALPHA, false>(s, V3(r.origin[0], r.origin[1], r.origin[2]),
                                 V3(r.direction[0], r.direction[1], r.direction[2]), r.tmin, r.tmax, hit, decal, st);
    out[i] = toPtHit(s, hit);
}

template <bool ALPHA> __global__ void k_trace_occlusion(DeviceScene s, const pt_ray *rays, uint64_t n, uint8_t *out)
{
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n)
        return;
    const pt_ray r = rays[i];
    Hit hit;
    Decal decal;
    TraversalStats st;
    traverse<false, ALPHA, false>(s, V3(r.origin[0], r.origin[1], r.origin[2]),
                                  V3(r.direction[0], r.direction[1], r.direction[2]), r.tmin, r.tmax, hit, decal, st);
    out[i] = hit.tri != 0xffffffffu;
}

CameraMatrices toCamera(const pt_render_params *p)
{
    CameraMatrices c;
    std::memcpy(c.view, p->view_inverse, 64);
    std::memcpy(c.proj, p->proj_inverse, 64);
    return c;
}

} // namespace

// ---------------------------------------------------------------------------------------------
// host drivers
// ---------------------------------------------------------------------------------------------
pt_status allocSortTemp(Context *ctx, size_t slots)
{
    size_t bytes = 0;
    PT_CUDA_CHECK(ctx, cub::DeviceRadixSort::SortPairs(nullptr, bytes, (const uint32_t *)nullptr, (uint32_t *)nullptr,
                                                       (const uint32_t *)nullptr, (uint32_t *)nullptr, (int)slots, 0, 32,
                                                       ctx->stream));
    bytes = (std::max<size_t>(bytes, 16) + 255) & ~(size_t)255;
    cudaFree(ctx->sortTemp);
    ctx->sortTemp = nullptr;
    ctx->sortTempBytes = 0;
    // one scratch area per pool (a pool never sorts more than all slots)
    PT_CUDA_CHECK(ctx, cudaMalloc(&ctx->sortTemp, bytes * PT_MAX_POOLS));
    ctx->sortTempBytes = bytes;
    return PT_OK;
}

// ---- pixel list of the tile set: 8x4 pixel blocks, so that consecutive work items are
//      neighbouring pixels and a warp's fresh primary rays are coherent -----------------------
static pt_status buildPixelList(Context *ctx, const pt_tile *tiles, uint32_t tileCount)
{
    const uint32_t W = ctx->width, H = ctx->height;
    const pt_tile whole = { 0, 0, W, H };
    std::vector<pt_tile> want(tileCount ? tiles : &whole, tileCount ? tiles + tileCount : &whole + 1);
    const bool same = ctx->pixelListValid && want.size() == ctx->pixelTiles.size() &&
                      (want.empty() || std::memcmp(want.data(), ctx->pixelTiles.data(), want.size() * sizeof(pt_tile)) == 0);
    if (!same)
    {
        // the tiles must be disjoint: a pixel listed twice would be sampled twice and k_resolve would race on it.
        // The total area is checked BEFORE any pixel is listed (many large tiles cannot exhaust host memory),
        // overlap with one bit per pixel while listing.
        uint64_t area = 0;
        for (const pt_tile &in : want)
        {
            const pt_tile t = { std::min(in.x0, W), std::min(in.y0, H), std::min(in.x1, W), std::min(in.y1, H) };
            if (t.x1 > t.x0 && t.y1 > t.y0)
                area += (uint64_t)(t.x1 - t.x0) * (t.y1 - t.y0);
            if (area > (uint64_t)W * H)
                return fail(ctx, PT_ERR_INVALID_ARGUMENT, "pt_render_samples", "tiles overlap (their area exceeds the frame)");
        }
        std::vector<uint32_t> list;
        list.reserve((size_t)area);
        std::vector<bool> covered((size_t)W * H, false);
        for (const pt_tile &in : want)
        {
            const pt_tile t = { std::min(in.x0, W), std::min(in.y0, H), std::min(in.x1, W), std::min(in.y1, H) };
            for (uint32_t y = t.y0; y < t.y1; y++)
                for (uint32_t x = t.x0; x < t.x1; x++)
                {
                    if (covered[(size_t)y * W + x])
                        return fail(ctx, PT_ERR_INVALID_ARGUMENT, "pt_render_samples", "tiles overlap");
                    covered[(size_t)y * W + x] = true;
                }
            for (uint32_t by = t.y0; by < t.y1; by += 4)
                for (uint32_t bx = t.x0; bx < t.x1; bx += 8)
                    for (uint32_t y = by; y < std::min(by + 4, t.y1); y++)
                        for (uint32_t x = bx; x < std::min(bx + 8, t.x1); x++)
                            list.push_back(y * W + x);
        }
        if (!list.empty())
            PT_CUDA_CHECK(ctx, cudaMemcpyAsync(ctx->pixelList, list.data(), list.size() * 4, cudaMemcpyHostToDevice,
                                               ctx->stream));
        PT_CUDA_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
        ctx->pixelTiles = want;
        ctx->pixelCount = (uint32_t)list.size();
        ctx->pixelListValid = true;
    }
    return PT_OK;
}

pt_status renderFrames(Context *ctx, const pt_render_params *params, uint32_t firstSample, uint32_t sampleCount, uint32_t samplesPerFrame,
                        const pt_tile *tiles, uint32_t tileCount)
{
    if (!params)
        return fail(ctx, PT_ERR_INVALID_ARGUMENT, "pt_render_samples", "params is NULL");
    if (!ctx->hasScene)
        return fail(ctx, PT_ERR_NO_SCENE, "pt_render_samples", "no scene uploaded");
    if (!ctx->accum)
        return fail(ctx, PT_ERR_NO_TARGET, "pt_render_samples", "pt_render_begin has not been called");
    if (params->bounce_count == 0 || params->bounce_count > 255)
        return fail(ctx, PT_ERR_INVALID_ARGUMENT, "pt_render_samples", "bounce_count must be in 1..255");
    if (samplesPerFrame == 0 || samplesPerFrame > kMaxSamplesPerFrame)
        return fail(ctx, PT_ERR_INVALID_ARGUMENT, "pt_render_frames", "samples_per_frame must be in 1..8192");
    if (ctx->targetContent == Context::TargetContent::Adaptive)
        return fail(ctx, PT_ERR_INVALID_ARGUMENT, "pt_render_samples",
                    "the target holds an adaptive render (per-pixel sample counts); call pt_render_begin first");
    if (tiles == nullptr)
        tileCount = 0;
    if (ctx->lightSampling == PT_LIGHT_SAMPLING_EMISSIVE_MIS && !ctx->emittersValid)
    {
        const pt_status st = buildEmitters(ctx);
        if (st != PT_OK)
            return st;
    }

    const pt_status listed = buildPixelList(ctx, tiles, tileCount);
    if (listed != PT_OK)
        return listed;
    if (sampleCount > 0)
        ctx->targetContent = Context::TargetContent::Uniform;
    uint32_t roundMax = 0;
    pt_status st = sizeSampleBuffer(ctx, sampleCount, roundMax);
    if (st == PT_OK)
        st = resetRenderStats(ctx);
    if (st == PT_OK)
        st = renderRounds(ctx, params, firstSample, sampleCount, samplesPerFrame, roundMax, false);
    return st == PT_OK ? finishRender(ctx, "pt_render_samples") : st;
}

pt_status sizeSampleBuffer(Context *ctx, uint32_t sampleCount, uint32_t &roundMax)
{
    const uint32_t pixels = ctx->pixelCount;
    // ---- rounds: as many samples per round as the sample buffer budget allows ---------------------
    roundMax = 0;
    if (pixels > 0 && sampleCount > 0)
    {
        size_t freeB = 0, totalB = 0;
        PT_CUDA_CHECK(ctx, cudaMemGetInfo(&freeB, &totalB));
        const uint64_t have = ctx->sbufCapacity * sizeof(float4);
        const uint64_t budget = std::max<uint64_t>(have, std::min<uint64_t>(ctx->sbufBudgetBytes, (freeB + have) / 2));
        // item indices are 32-bit
        const uint64_t maxItems = std::min<uint64_t>(budget / sizeof(float4), 0xfffffff0ull);
        roundMax = (uint32_t)std::min<uint64_t>(sampleCount, std::max<uint64_t>(1, maxItems / pixels));
        const uint64_t need = (uint64_t)roundMax * pixels;
        if (need > ctx->sbufCapacity)
        {
            PT_CUDA_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
            cudaFree(ctx->sbuf);
            ctx->sbuf = nullptr;
            ctx->sbufCapacity = 0;
            PT_CUDA_CHECK(ctx, cudaMalloc((void **)&ctx->sbuf, need * sizeof(float4)));
            ctx->sbufCapacity = need;
        }
    }
    return PT_OK;
}

pt_status resetRenderStats(Context *ctx)
{
    ctx->stats.kernel_launches = 0;
    ctx->stats.wavefront_iterations = 0;
    for (int k = 0; k < PT_KERNEL_CLASS_COUNT; k++)
    {
        ctx->stats.kernel_ms[k] = 0.0f;
        ctx->stats.kernel_launch_count[k] = 0;
    }
    PT_CUDA_CHECK(ctx, cudaMemsetAsync(ctx->dCounters, 0, sizeof(DeviceCounters), ctx->stream));
    PT_CUDA_CHECK(ctx, cudaEventRecord(ctx->evStart, ctx->stream));
    return PT_OK;
}

pt_status renderRounds(Context *ctx, const pt_render_params *params, uint32_t firstSample, uint32_t sampleCount, uint32_t samplesPerFrame,
                       uint32_t roundMax, bool adaptive)
{
    const uint32_t W = ctx->width, H = ctx->height;
    const uint32_t pixels = ctx->pixelCount;

    // optional per-launch CUDA-event timing (pt_set_kernel_timing): (class, start, stop) triples
    struct Timed
    {
        int cls;
        cudaEvent_t a, b;
    };
    std::vector<Timed> timed;
    // every path out of this function — PT_CUDA_CHECK returns early on an error — destroys the timing events still
    // alive and, if the render did not finish, waits for what the pools' streams were already given
    bool finished = false;
    struct Cleanup
    {
        Context *ctx;
        std::vector<Timed> &timed;
        bool &finished;
        ~Cleanup()
        {
            for (Timed &t : timed)
            {
                if (t.a)
                    cudaEventDestroy(t.a);
                if (t.b)
                    cudaEventDestroy(t.b);
            }
            timed.clear();
            if (!finished)
            {
                for (int i = 0; i < PT_MAX_POOLS; i++)
                    if (ctx->poolStreams[i])
                        cudaStreamSynchronize(ctx->poolStreams[i]);
                cudaStreamSynchronize(ctx->stream);
                cudaGetLastError();
            }
        }
    } cleanup { ctx, timed, finished };
    const bool timing = ctx->kernelTiming;
    auto begin = [&](int cls, cudaStream_t st) {
        if (!timing)
            return;
        Timed t { cls, nullptr, nullptr };
        cudaEventCreate(&t.a);
        cudaEventCreate(&t.b);
        cudaEventRecord(t.a, st);
        timed.push_back(t);
        ctx->stats.kernel_launch_count[cls]++;
    };
    auto end = [&](cudaStream_t st) {
        if (timing)
            cudaEventRecord(timed.back().b, st);
    };

    const bool alpha = ctx->scene.hasAlpha != 0;
    const bool statsOn = ctx->collectTraversalStats;
    // emissive-MIS light sampling: without emitters it is the reference mode, which k_shade renders bit for bit
    const bool emissive = ctx->lightSampling == PT_LIGHT_SAMPLING_EMISSIVE_MIS && ctx->emitters.count > 0;
    EmitterTable emitters = ctx->emitters;
    {
        // the emitter branch's probability: 1 when no analytic light can contribute, 1/2 otherwise
        const LightBlock &lb = ctx->hostLights;
        const bool analytic = lb.count > 0 || lb.dirColor.x != 0.0f || lb.dirColor.y != 0.0f || lb.dirColor.z != 0.0f;
        emitters.pEmitter = analytic ? 0.5f : 1.0f;
    }
    // Hits are shaded in triangle order (radix sort of the hit queue on the upper bits of the
    // leaf-order = Morton-order triangle index): neighbouring lanes then shade neighbouring
    // triangles — same material branch, same texture region, shared cache lines.  16 key bits
    // are plenty for that.
    uint32_t triBits = 1;
    while (triBits < 32 && (ctx->scene.triCount >> triBits) != 0)
        triBits++;
    const uint32_t keyBits = std::min(triBits, (uint32_t)PT_HIT_KEY_BITS);

    for (uint32_t roundBase = 0; roundMax > 0 && roundBase < sampleCount; roundBase += roundMax)
    {
        RenderConst base = {};
        base.scene = ctx->scene;
        base.cam = toCamera(params);
        base.accum = ctx->accum;
        base.counters = ctx->dCounters;
        base.width = W;
        base.height = H;
        base.firstSample = firstSample;
        base.sampleCount = sampleCount;
        base.samplesPerFrame = samplesPerFrame;
        base.bounceCount = params->bounce_count;
        base.lensRadius = params->lens_radius;
        base.focalDistance = params->focal_distance;
        base.missFlags = params->miss_flags;
        base.hitFlags = params->hit_flags;
        base.pixelList = ctx->pixelList;
        base.pixelCount = pixels;
        base.sbuf = ctx->sbuf;
        base.roundBase = roundBase;
        base.roundSamples = std::min(roundMax, sampleCount - roundBase);
        base.itemCount = base.roundSamples * pixels;
        base.nextItem = ctx->dNextItem;
        base.hitKeyShift = triBits - keyBits;

        // ---- pools: independent sub-wavefronts on their own streams ------------------------------
        // A traversal kernel ends with its longest rays (a ray grazing the tessellated board visits
        // thousands of nodes); with one wavefront the whole GPU waits for them every iteration.
        // Several smaller wavefronts on separate streams fill those tails with each other's kernels.
        const uint32_t slotsTotal = std::min(ctx->slotCapacity, base.itemCount);
        uint32_t poolCount = std::max(1u, std::min(ctx->poolCount, slotsTotal / 16384u));
        const uint32_t poolSlots = slotsTotal / poolCount; // the last pool takes the remainder
        struct Pool
        {
            RenderConst rc;
            cudaStream_t stream;
            QueueCounts *hq;
            void *sortTemp;
            uint32_t gridExtend, gridShadow, gridShade, gridWide;
            int cur;
            bool active;
        };
        std::vector<Pool> pools(poolCount);
        PT_CUDA_CHECK(ctx, cudaMemcpyAsync(ctx->dNextItem, &slotsTotal, 4, cudaMemcpyHostToDevice, ctx->stream));
        PT_CUDA_CHECK(ctx, cudaEventRecord(ctx->evRound, ctx->stream));
        for (uint32_t p = 0; p < poolCount; p++)
        {
            Pool &pl = pools[p];
            const uint32_t first = p * poolSlots;
            const uint32_t slots = p + 1 == poolCount ? slotsTotal - first : poolSlots;
            pl.rc = base;
            pl.rc.ps = ctx->ps;
            // queues are private to the pool: its sub-range of the queue arrays
            pl.rc.ps.contQ[0] += first, pl.rc.ps.contQ[1] += first;
            pl.rc.ps.regenQ[0] += first, pl.rc.ps.regenQ[1] += first;
            pl.rc.ps.hitQ += first, pl.rc.ps.hitKey += first;
            pl.rc.ps.hitQSorted += first, pl.rc.ps.hitKeySorted += first, pl.rc.ps.shadowQueue += first;
            pl.rc.qc = ctx->dQueueCounts + p;
            pl.rc.slotBase = first;
            pl.rc.slotCount = slots;
            pl.rc.sortHits = ctx->sortHits && slots >= 4096;
            pl.stream = poolCount == 1 ? ctx->stream : ctx->poolStreams[p];
            pl.hq = ctx->hQueueCounts + p;
            pl.sortTemp = (char *)ctx->sortTemp + p * ctx->sortTempBytes;
            pl.cur = 0;
            pl.active = true;
            pl.gridShade = std::min((slots + 127) / 128, (uint32_t)ctx->smCount * PT_SHADE_GRID_PER_SM);
            // persistent warps: exactly as many blocks as are resident on the machine (occupancy query per
            // instantiation; PT_TRACE_BLOCKS overrides), never more than the rays need
            auto residentGrid = [&](auto kernel) {
                int perSM = 0;
                if (ctx->traceBlocksPerSM)
                    perSM = (int)ctx->traceBlocksPerSM;
                else if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&perSM, kernel, 128, 0) != cudaSuccess || perSM < 1)
                    perSM = 4;
                return std::min((slots + 127) / 128, (uint32_t)(ctx->smCount * perSM));
            };
            if (alpha && statsOn)
                pl.gridExtend = residentGrid(k_extend<true, true>), pl.gridShadow = residentGrid(k_shadow<true, true>);
            else if (alpha)
                pl.gridExtend = residentGrid(k_extend<true, false>), pl.gridShadow = residentGrid(k_shadow<true, false>);
            else if (statsOn)
                pl.gridExtend = residentGrid(k_extend<false, true>), pl.gridShadow = residentGrid(k_shadow<false, true>);
            else
                pl.gridExtend = residentGrid(k_extend<false, false>), pl.gridShadow = residentGrid(k_shadow<false, false>);
            pl.gridWide = std::min((slots + 255) / 256, (uint32_t)ctx->smCount * 8);
            if (pl.stream != ctx->stream)
                PT_CUDA_CHECK(ctx, cudaStreamWaitEvent(pl.stream, ctx->evRound, 0));
            k_init<<<pl.gridWide, 256, 0, pl.stream>>>(pl.rc);
            ctx->stats.kernel_launches++;
        }

        auto iteration = [&](Pool &pl) -> pt_status {
            const RenderConst &rc = pl.rc;
            const int cur = pl.cur;
            cudaStream_t st = pl.stream;
            // launches KERNEL<alpha, statsOn, ...> ARGS: the runtime flags as template arguments, then the arguments that
            // follow ARGS, if any (", ##" drops the comma when there are none)
#define PT_DISPATCH(KERNEL, GRID, BLOCK, ARGS, ...)                                                                   \
    do                                                                                                                \
    {                                                                                                                 \
        if (alpha && statsOn)                                                                                         \
            KERNEL<true, true, ##__VA_ARGS__><<<GRID, BLOCK, 0, st>>> ARGS;                                           \
        else if (alpha)                                                                                               \
            KERNEL<true, false, ##__VA_ARGS__><<<GRID, BLOCK, 0, st>>> ARGS;                                          \
        else if (statsOn)                                                                                             \
            KERNEL<false, true, ##__VA_ARGS__><<<GRID, BLOCK, 0, st>>> ARGS;                                          \
        else                                                                                                          \
            KERNEL<false, false, ##__VA_ARGS__><<<GRID, BLOCK, 0, st>>> ARGS;                                         \
    } while (0)
            begin(PT_KERNEL_EXTEND, st);
            if (rc.sortHits)
                PT_CUDA_CHECK(ctx, cudaMemsetAsync(rc.ps.hitKey, 0xff, (size_t)rc.slotCount * 4, st));
            PT_DISPATCH(k_extend, pl.gridExtend, 128, (rc, cur));
            end(st);
            begin(PT_KERNEL_SHADE, st);
            if (rc.sortHits)
            {
                // unused tail of the key array sorts to the end (k_shade only reads qc->hit entries)
                size_t bytes = ctx->sortTempBytes;
                PT_CUDA_CHECK(ctx, cub::DeviceRadixSort::SortPairs(pl.sortTemp, bytes, rc.ps.hitKey, rc.ps.hitKeySorted,
                                                                   rc.ps.hitQ, rc.ps.hitQSorted, (int)rc.slotCount, 0,
                                                                   (int)keyBits + 1, st));
            }
            if (emissive)
                PT_DISPATCH(k_shade, pl.gridShade, 128, (rc, cur, emitters), true);
            else
                PT_DISPATCH(k_shade, pl.gridShade, 128, (rc, cur, emitters), false);
            end(st);
            begin(PT_KERNEL_SHADOW, st);
            PT_DISPATCH(k_shadow, pl.gridShadow, 128, (rc, cur));
            end(st);
#undef PT_DISPATCH
            ctx->stats.kernel_launches += 3;
            pl.cur ^= 1;
            return PT_OK;
        };

        // the host polls the queue sizes every few iterations; a round needs at least
        // items / slots iterations, so polling starts sparse and gets denser towards the end
        uint32_t checkEvery = 4;
        for (uint32_t live = poolCount; live > 0;)
        {
            for (uint32_t k = 0; k < checkEvery; k++)
            {
                for (Pool &pl : pools)
                    if (pl.active)
                    {
                        const pt_status st = iteration(pl);
                        if (st != PT_OK)
                            return st;
                    }
                ctx->stats.wavefront_iterations++;
            }
            for (Pool &pl : pools)
                if (pl.active)
                    PT_CUDA_CHECK(ctx, cudaMemcpyAsync(pl.hq, pl.rc.qc, sizeof(QueueCounts), cudaMemcpyDeviceToHost, pl.stream));
            bool first = true;
            for (Pool &pl : pools)
                if (pl.active)
                {
                    if (first)
                        PT_CUDA_CHECK(ctx, cudaMemcpyAsync(ctx->hNextItem, ctx->dNextItem, 4, cudaMemcpyDeviceToHost, pl.stream));
                    first = false;
                    PT_CUDA_CHECK(ctx, cudaStreamSynchronize(pl.stream));
                    if (pl.hq->cont[pl.cur] + pl.hq->regen[pl.cur] == 0)
                    {
                        pl.active = false;
                        live--;
                    }
                }
            // while work items remain, at least remaining / slots more iterations are needed
            const uint32_t nextItem = *ctx->hNextItem;
            const uint64_t remaining = nextItem < base.itemCount ? base.itemCount - nextItem : 0;
            checkEvery = (uint32_t)std::min<uint64_t>(64, std::max<uint64_t>(4, remaining / std::max(1u, slotsTotal)));
        }
        // every pool has been synchronised with the host: the round's samples are all parked
        begin(PT_KERNEL_FINISH, ctx->stream);
        const uint32_t resolveGrid = std::min((pixels + 255) / 256, (uint32_t)ctx->smCount * 8);
        if (adaptive)
            k_resolve<true><<<resolveGrid, 256, 0, ctx->stream>>>(base, ctx->adaptivePixels);
        else
            k_resolve<false><<<resolveGrid, 256, 0, ctx->stream>>>(base, nullptr);
        end(ctx->stream);
        ctx->stats.kernel_launches++;
    }
    if (timing)
    {
        cudaDeviceSynchronize();
        for (Timed &t : timed)
        {
            float ms = 0.0f;
            cudaEventElapsedTime(&ms, t.a, t.b);
            ctx->stats.kernel_ms[t.cls] += ms;
        }
    }
    // what is still queued runs on ctx->stream only: every pool has been synchronised with the host
    finished = true;
    return PT_OK;
}

pt_status finishRender(Context *ctx, const char *what)
{
    PT_CUDA_CHECK(ctx, cudaEventRecord(ctx->evStop, ctx->stream));
    PT_CUDA_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    PT_CUDA_CHECK(ctx, cudaGetLastError());
    PT_CUDA_CHECK(ctx, cudaEventElapsedTime(&ctx->stats.last_render_ms, ctx->evStart, ctx->evStop));
    return checkStackOverflow(ctx, what);
}

pt_status checkStackOverflow(Context *ctx, const char *what)
{
    unsigned int n = 0;
    PT_CUDA_CHECK(ctx, cudaMemcpyFromSymbol(&n, g_stackOverflows, sizeof(n)));
    if (n == 0)
        return PT_OK;
    const unsigned int zero = 0;
    cudaMemcpyToSymbol(g_stackOverflows, &zero, sizeof(zero));
    ctx->stats.stack_overflows = n;
    char buf[192];
    std::snprintf(buf, sizeof(buf), "the traversal stack (%d entries) overflowed %u times on a BVH of depth %u: sub-trees were "
                                    "skipped, the result is not valid", PT_STACK_SIZE, n, ctx->bvhMaxDepth);
    return fail(ctx, PT_ERR_UNSUPPORTED, what, buf);
}

pt_status firstHitAov(Context *ctx, const pt_render_params *params, uint32_t width, uint32_t height, pt_hit *out)
{
    if (!params || !out || width == 0 || height == 0)
        return fail(ctx, PT_ERR_INVALID_ARGUMENT, "pt_first_hit_aov", "bad argument");
    if (!ctx->hasScene)
        return fail(ctx, PT_ERR_NO_SCENE, "pt_first_hit_aov", "no scene uploaded");
    const size_t n = (size_t)width * height;
    pt_hit *dOut = nullptr;
    PT_CUDA_CHECK(ctx, cudaMalloc((void **)&dOut, n * sizeof(pt_hit)));
    const uint32_t grid = (uint32_t)((n + 127) / 128);
    if (ctx->scene.hasAlpha)
        k_first_hit<true><<<grid, 128, 0, ctx->stream>>>(ctx->scene, toCamera(params), width, height, dOut);
    else
        k_first_hit<false><<<grid, 128, 0, ctx->stream>>>(ctx->scene, toCamera(params), width, height, dOut);
    cudaError_t err = cudaMemcpyAsync(out, dOut, n * sizeof(pt_hit), cudaMemcpyDeviceToHost, ctx->stream);
    if (err == cudaSuccess)
        err = cudaStreamSynchronize(ctx->stream);
    cudaFree(dOut);
    PT_CUDA_CHECK(ctx, err);
    return checkStackOverflow(ctx, "pt_first_hit_aov");
}

pt_status debugRender(Context *ctx, const pt_render_params *params, const pt_debug_params *dbg, uint32_t width, uint32_t height,
                      float *out)
{
    if (!params || !dbg || !out || width == 0 || height == 0 || dbg->render_mode > PT_DEBUG_MODE_INSTANCE)
        return fail(ctx, PT_ERR_INVALID_ARGUMENT, "pt_debug_render", "bad argument");
    if (!ctx->hasScene)
        return fail(ctx, PT_ERR_NO_SCENE, "pt_debug_render", "no scene uploaded");
    const size_t n = (size_t)width * height;
    float4 *dOut = nullptr;
    PT_CUDA_CHECK(ctx, poolAlloc(ctx, (void **)&dOut, n * sizeof(float4), ctx->stream));
    const uint32_t grid = (uint32_t)((n + 127) / 128);
    const bool alphaScene = ctx->scene.hasAlpha != 0;
    const bool alphaPrimary = alphaScene && !(dbg->raygen_flags & PT_DEBUG_RAYGEN_FORCE_OPAQUE);
    const CameraMatrices cam = toCamera(params);
    const bool cull = (dbg->raygen_flags & PT_DEBUG_RAYGEN_CULL_BACK_FACES) != 0;
#define PT_DEBUG_LAUNCH(AP, AS)                                                                                       \
    do                                                                                                                \
    {                                                                                                                 \
        if (cull)                                                                                                     \
            k_debug<AP, AS, true><<<grid, 128, 0, ctx->stream>>>(ctx->scene, cam, width, height, params->miss_flags, *dbg, dOut); \
        else                                                                                                          \
            k_debug<AP, AS, false><<<grid, 128, 0, ctx->stream>>>(ctx->scene, cam, width, height, params->miss_flags, *dbg, dOut); \
    } while (0)
    if (alphaPrimary)
        PT_DEBUG_LAUNCH(true, true);
    else if (alphaScene)
        PT_DEBUG_LAUNCH(false, true);
    else
        PT_DEBUG_LAUNCH(false, false);
#undef PT_DEBUG_LAUNCH
    cudaError_t err = cudaGetLastError();
    if (err == cudaSuccess)
        err = cudaMemcpyAsync(out, dOut, n * sizeof(float4), cudaMemcpyDeviceToHost, ctx->stream);
    if (err == cudaSuccess)
        err = cudaStreamSynchronize(ctx->stream);
    cudaFreeAsync(dOut, ctx->stream);
    PT_CUDA_CHECK(ctx, err);
    return checkStackOverflow(ctx, "pt_debug_render");
}

void launchDenoiseGuides(Context *ctx, const pt_render_params *params, float4 *albedoT, float4 *normal)
{
    const uint32_t width = ctx->width, height = ctx->height;
    const uint32_t grid = (uint32_t)(((size_t)width * height + 127) / 128);
    const uint32_t flags = (params->hit_flags & PT_HIT_FLAGS_DX_NORMAL_TEXTURES) ? PT_DEBUG_HIT_DX_NORMAL_TEXTURES : 0u;
    if (ctx->scene.hasAlpha)
        k_denoise_guides<true><<<grid, 128, 0, ctx->stream>>>(ctx->scene, toCamera(params), width, height, flags, albedoT, normal);
    else
        k_denoise_guides<false><<<grid, 128, 0, ctx->stream>>>(ctx->scene, toCamera(params), width, height, flags, albedoT, normal);
}

pt_status traceClosest(Context *ctx, const pt_ray *rays, uint64_t n, pt_hit *out)
{
    if ((n && (!rays || !out)))
        return fail(ctx, PT_ERR_INVALID_ARGUMENT, "pt_trace_closest", "bad argument");
    if (!ctx->hasScene)
        return fail(ctx, PT_ERR_NO_SCENE, "pt_trace_closest", "no scene uploaded");
    if (n == 0)
        return PT_OK;
    pt_ray *dRays = nullptr;
    pt_hit *dOut = nullptr;
    PT_CUDA_CHECK(ctx, cudaMalloc((void **)&dRays, n * sizeof(pt_ray)));
    cudaError_t err = cudaMalloc((void **)&dOut, n * sizeof(pt_hit));
    if (err == cudaSuccess)
        err = cudaMemcpyAsync(dRays, rays, n * sizeof(pt_ray), cudaMemcpyHostToDevice, ctx->stream);
    if (err == cudaSuccess)
    {
        const uint32_t grid = (uint32_t)((n + 127) / 128);
        if (ctx->scene.hasAlpha)
            k_trace_closest<true><<<grid, 128, 0, ctx->stream>>>(ctx->scene, dRays, n, dOut);
        else
            k_trace_closest<false><<<grid, 128, 0, ctx->stream>>>(ctx->scene, dRays, n, dOut);
        err = cudaMemcpyAsync(out, dOut, n * sizeof(pt_hit), cudaMemcpyDeviceToHost, ctx->stream);
    }
    if (err == cudaSuccess)
        err = cudaStreamSynchronize(ctx->stream);
    cudaFree(dRays);
    cudaFree(dOut);
    PT_CUDA_CHECK(ctx, err);
    return checkStackOverflow(ctx, "pt_trace_closest");
}

pt_status traceOcclusion(Context *ctx, const pt_ray *rays, uint64_t n, uint8_t *out)
{
    if ((n && (!rays || !out)))
        return fail(ctx, PT_ERR_INVALID_ARGUMENT, "pt_trace_occlusion", "bad argument");
    if (!ctx->hasScene)
        return fail(ctx, PT_ERR_NO_SCENE, "pt_trace_occlusion", "no scene uploaded");
    if (n == 0)
        return PT_OK;
    pt_ray *dRays = nullptr;
    uint8_t *dOut = nullptr;
    PT_CUDA_CHECK(ctx, cudaMalloc((void **)&dRays, n * sizeof(pt_ray)));
    cudaError_t err = cudaMalloc((void **)&dOut, n);
    if (err == cudaSuccess)
        err = cudaMemcpyAsync(dRays, rays, n * sizeof(pt_ray), cudaMemcpyHostToDevice, ctx->stream);
    if (err == cudaSuccess)
    {
        const uint32_t grid = (uint32_t)((n + 127) / 128);
        if (ctx->scene.hasAlpha)
            k_trace_occlusion<true><<<grid, 128, 0, ctx->stream>>>(ctx->scene, dRays, n, dOut);
        else
            k_trace_occlusion<false><<<grid, 128, 0, ctx->stream>>>(ctx->scene, dRays, n, dOut);
        err = cudaMemcpyAsync(out, dOut, n, cudaMemcpyDeviceToHost, ctx->stream);
    }
    if (err == cudaSuccess)
        err = cudaStreamSynchronize(ctx->stream);
    cudaFree(dRays);
    cudaFree(dOut);
    PT_CUDA_CHECK(ctx, err);
    return checkStackOverflow(ctx, "pt_trace_occlusion");
}

} // namespace pt
