// scene.cuh — device-resident scene layout (HBM) and the software texture sampler.
//
// Layout, designed for the traversal / shade kernels rather than copied from the reference:
//   * instances x meshes are FLATTENED at upload: every instanced triangle is baked to world
//     space once (the reference re-derives the 4x4 transform and inverts it four times per hit,
//     PT/Shaders/sampling.glsl:5-15).  Flattened triangle id order = instance, mesh-in-model,
//     primitive (this id breaks ties in t, so results do not depend on the BVH).
//   * triangles are stored in two streams:
//       TriPos   48 B  — three float4 per BVH reference, in BVH leaf order: world positions, .w lanes carry
//                        flat id / flags / material id; read by the intersection loop (coalesced 16-B loads);
//       TriShade 192 B — twelve float4 per triangle, in flattened order, reached through the flat id:
//                        world normals / tangents / bitangents of the three corners, the three UVs, the
//                        (instance, geometry, primitive) triple and the unit normals; read once per shaded hit.
//   * wide BVH nodes are 64 B: child boxes quantised to 8 bits per plane + 4 child references.
//   * textures: RGBA8 (or float) mip chains, one allocation per texture, sampled in software (bilinear x
//     trilinear, repeat) so that CPU oracle and GPU agree; sRGB decode through a 256-entry LUT.
#pragma once
#include "vecmath.cuh"

namespace pt
{

// ---------------------------------------------------------------------------------------------
// BVH4 node, 64 bytes: the child boxes quantised to 8 bits per plane on a per-node grid (origin = min corner of
// the node, one power-of-two step per axis; Ylitie, Karras, Laine 2017 in 4-wide form), rounded OUTWARDS so that a
// quantised box always contains the exact one: traversal stays conservative, hits are unchanged, and a node costs
// half the cache footprint of fp32 boxes (the trace kernels live on L1 / L2 capacity for nodes, DESIGN.md §3).
// ---------------------------------------------------------------------------------------------
struct __align__(16) BvhNode
{
    float ox, oy, oz; // grid origin
    float sx;         // grid steps (powers of two)
    float sy, sz;
    uint32_t qlox, qloy; // byte i of q* = plane of child i in grid steps from the origin
    uint32_t qloz, qhix, qhiy, qhiz;
    int4 child; // >= 0: internal node index; < 0: leaf, ~child = (firstTri << 2) | (count - 1)
};
static_assert(sizeof(BvhNode) == 64, "quantised BvhNode must be 64 bytes");

#define PT_CHILD_EMPTY 0x7fffffff
#define PT_MAX_LEAF_TRIS 4 // the leaf code has two bits for the count

PT_HD int encodeLeaf(uint32_t first, uint32_t count) { return ~(int)((first << 2) | (count - 1)); }

#define PT_TRI_FLAG_OPAQUE 1u
#define PT_TRI_FLAG_MIRRORED 2u // the instance transform has a negative determinant: object-space winding = world-space winding reversed

// The shading records stay in FLATTENED triangle order and are reached through the flat id a leaf entry carries
// (__float_as_uint(triPos[3 * k].w)): one record per triangle however many references the BVH holds to it.
struct __align__(16) TriShade
{
    float4 a[12];
    // a[0] = n0.xyz, n1.x   a[1] = n1.yz, n2.xy   a[2] = n2.z, t0.xyz
    // a[3] = t1.xyz, t2.x   a[4] = t2.yz, b0.xy   a[5] = b0.z, b1.xyz
    // a[6] = b2.xyz, uv0.x  a[7] = uv0.y, uv1.xy, uv2.x   a[8] = uv2.y, instance, geometry, primitive (bits)
    // a[9] = normalize(n0).xyz, normalize(n1).x   a[10] = normalize(n1).yz, normalize(n2).xy
    // a[11] = normalize(n2).z, normalize(cross(p1 - p0, p2 - p0)).xyz — what k_shade would normalise per HIT, normalised
    //         once per TRIANGLE by k_bake with the same device functions on the same values (closestHit.rchit:60-66,
    //         76-78), so the bits are those of the per-hit evaluation
};
static_assert(sizeof(TriShade) == 192, "TriShade must be 192 bytes");

// ---------------------------------------------------------------------------------------------
// materials: the reference's 96-byte structs, verbatim (PT/Shaders/ShaderTypes.incl:61-118)
// ---------------------------------------------------------------------------------------------
struct __align__(16) MaterialRaw
{
    float4 q[6];
};

// ---------------------------------------------------------------------------------------------
// textures
// ---------------------------------------------------------------------------------------------
#define PT_MAX_TEX_LEVELS 16
#define PT_TEX_FLAG_SRGB 1u
#define PT_TEX_FLAG_FLOAT 2u

struct DevTexture
{
    uint64_t base; // device address of level 0 (levels follow contiguously)
    uint32_t width, height;
    uint32_t levels;
    uint32_t flags;
    uint32_t levelOffset[PT_MAX_TEX_LEVELS]; // in texels, relative to base
};

struct LightBlock
{
    uint32_t count;
    uint32_t pad[3];
    float4 dirColor;     // DirectionalLight.Color
    float4 dirDirection; // DirectionalLight.Direction
    float4 point[64 * 3]; // PointLight: color|pad, position|pad, (c, l, q, pad)
};

struct DeviceScene
{
    const BvhNode *nodes;
    const float4 *triPos;     // 3 per BVH reference, leaf order
    const TriShade *triShade; // flattened order, indexed by the flat id
    const MaterialRaw *materials[3]; // by material type
    const DevTexture *textures;
    const float *lut; // [0..255] unorm, [256..511] sRGB -> linear
    const LightBlock *lights;
    DevTexture sky2D;
    uint32_t triCount;
    uint32_t textureCount;
    uint32_t hasAlpha; // any non-opaque triangle
    uint32_t hasSky2D;
    uint32_t skyCubeSlot; // first of six consecutive entries of textures[] (+X, -X, +Y, -Y, +Z, -Z); 0 = no cube sky
    uint32_t maxAnisotropy; // sampler state of textureGrad: 1 = isotropic trilinear .. 16 (pt_set_sampler)
};

// ---------------------------------------------------------------------------------------------
// sampler (linear / linear-mip / repeat / anisotropic — see oracle/pt_oracle.cpp for the definition)
// ---------------------------------------------------------------------------------------------
PT_DEV float4 fetchTexel(const DeviceScene &s, const DevTexture &t, uint32_t level, uint32_t x, uint32_t y, uint32_t lw)
{
    const size_t idx = (size_t)t.levelOffset[level] + (size_t)y * lw + x;
    if (t.flags & PT_TEX_FLAG_FLOAT)
        return __ldg(reinterpret_cast<const float4 *>(t.base) + idx);
    const uchar4 c = __ldg(reinterpret_cast<const uchar4 *>(t.base) + idx);
    const float *lut = s.lut + ((t.flags & PT_TEX_FLAG_SRGB) ? 256 : 0);
    return make_float4(__ldg(lut + c.x), __ldg(lut + c.y), __ldg(lut + c.z), __ldg(s.lut + c.w));
}

PT_DEV float4 lerp4(float4 a, float4 b, float f)
{
    const float g = 1.0f - f;
    return make_float4(a.x * g + b.x * f, a.y * g + b.y * f, a.z * g + b.z * f, a.w * g + b.w * f);
}

PT_DEV float4 sampleBilinear(const DeviceScene &s, const DevTexture &t, uint32_t level, float u, float v)
{
    const uint32_t lw = max(1u, t.width >> level), lh = max(1u, t.height >> level);
    if (lw == 1 && lh == 1)
        return fetchTexel(s, t, level, 0, 0, 1);
    u = isfinite(u) ? u : 0.0f;
    v = isfinite(v) ? v : 0.0f;
    u = u - floorf(u);
    v = v - floorf(v);
    const float x = u * (float)lw - 0.5f, y = v * (float)lh - 0.5f;
    const float fx0 = floorf(x), fy0 = floorf(y);
    const float fx = x - fx0, fy = y - fy0;
    const int W = (int)lw, H = (int)lh;
    // repeat wrap: u, v are in [0, 1] here, so floor(x) is in [-1, W - 1] and one conditional
    // replaces the oracle's ((i % W) + W) % W (same integers, no integer divisions)
    const int ix = (int)fx0, iy = (int)fy0;
    const int x0 = ix < 0 ? W - 1 : ix, x1 = x0 + 1 == W ? 0 : x0 + 1;
    const int y0 = iy < 0 ? H - 1 : iy, y1 = y0 + 1 == H ? 0 : y0 + 1;
    const float4 t00 = fetchTexel(s, t, level, x0, y0, lw), t10 = fetchTexel(s, t, level, x1, y0, lw);
    const float4 t01 = fetchTexel(s, t, level, x0, y1, lw), t11 = fetchTexel(s, t, level, x1, y1, lw);
    return lerp4(lerp4(t00, t10, fx), lerp4(t01, t11, fx), fy);
}

// texture() outside a fragment stage: level 0
PT_DEV float4 textureLod0(const DeviceScene &s, const DevTexture &t, float u, float v)
{
    return sampleBilinear(s, t, 0, u, v);
}

// texture(samplerCube, dir) outside a fragment stage: level 0, linear; Vulkan face selection
// (z wins ties over y over x), footprint clamped to the face — oracle/pt_oracle.cpp sampleCube
PT_DEV float4 sampleCube(const DeviceScene &s, uint32_t firstSlot, vec3 r)
{
    const float ax = fabsf(r.x), ay = fabsf(r.y), az = fabsf(r.z);
    uint32_t face;
    float sc, tc, ma;
    if (az >= ax && az >= ay)
    {
        face = r.z < 0.0f ? 5 : 4;
        sc = r.z < 0.0f ? -r.x : r.x;
        tc = -r.y;
        ma = az;
    }
    else if (ay >= ax)
    {
        face = r.y < 0.0f ? 3 : 2;
        sc = r.x;
        tc = r.y < 0.0f ? -r.z : r.z;
        ma = ay;
    }
    else
    {
        face = r.x < 0.0f ? 1 : 0;
        sc = r.x < 0.0f ? r.z : -r.z;
        tc = -r.y;
        ma = ax;
    }
    const DevTexture &t = s.textures[firstSlot + face];
    float u = 0.5f * (sc / ma + 1.0f), v = 0.5f * (tc / ma + 1.0f);
    u = isfinite(u) ? u : 0.5f;
    v = isfinite(v) ? v : 0.5f;
    const float x = u * (float)t.width - 0.5f, y = v * (float)t.height - 0.5f;
    const float fx0 = floorf(x), fy0 = floorf(y);
    const float fx = x - fx0, fy = y - fy0;
    const int W = (int)t.width, H = (int)t.height;
    const int x0 = min(max((int)fx0, 0), W - 1), x1 = min(max((int)fx0 + 1, 0), W - 1);
    const int y0 = min(max((int)fy0, 0), H - 1), y1 = min(max((int)fy0 + 1, 0), H - 1);
    const float4 t00 = fetchTexel(s, t, 0, x0, y0, t.width), t10 = fetchTexel(s, t, 0, x1, y0, t.width);
    const float4 t01 = fetchTexel(s, t, 0, x0, y1, t.width), t11 = fetchTexel(s, t, 0, x1, y1, t.width);
    return lerp4(lerp4(t00, t10, fx), lerp4(t01, t11, fx), fy);
}

// Footprint of a textureGrad lookup (Vulkan "Texel Anisotropic Filtering", the specification's example implementation;
// definition and citations in oracle/pt_oracle.cpp textureGrad): N taps along the major axis, all at level-of-detail
// lambda = log2(rho_max / eta).  Returns the lower mip level and the blend weight towards the next one (0 = one level).
struct GradFootprint
{
    uint32_t level; // lower level
    float frac;     // trilinear weight of level + 1
    uint32_t taps;  // N, 1 .. maxAnisotropy
    float du, dv;   // major-axis derivative (uv units)
};
PT_DEV GradFootprint gradFootprint(const DevTexture &t, float4 deriv, uint32_t maxAnisotropy)
{
    GradFootprint g;
    g.level = 0;
    g.frac = 0.0f;
    g.taps = 1;
    g.du = g.dv = 0.0f;
    const uint32_t last = t.levels - 1;
    if (last == 0)
        return g;
    const float w = (float)t.width, h = (float)t.height;
    const float ax = deriv.x * w, ay = deriv.y * h, bx = deriv.z * w, by = deriv.w * h;
    const float rx2 = ax * ax + ay * ay, ry2 = bx * bx + by * by;
    const float rho2 = fmaxf(rx2, ry2);
    float eta = 1.0f;
    if (maxAnisotropy > 1 && rho2 > 0.0f)
    {
        const float rmin2 = fminf(rx2, ry2);
        const float ratio = sqrtf(rho2) / sqrtf(rmin2);
        eta = (ratio <= (float)maxAnisotropy) ? fmaxf(ratio, 1.0f) : (float)maxAnisotropy;
        g.taps = (uint32_t)ceilf(eta);
        if (rx2 > ry2)
            g.du = deriv.x, g.dv = deriv.y;
        else
            g.du = deriv.z, g.dv = deriv.w;
    }
    const float lambda = 0.5f * log2f(rho2 / (eta * eta));
    if (!(lambda > 0.0f))
        return g;
    if (lambda >= (float)last)
    {
        g.level = last;
        g.taps = 1; // at the 1 x 1 top level every tap reads the same texel
        return g;
    }
    const float fl = floorf(lambda);
    g.frac = lambda - fl;
    g.level = (uint32_t)fl;
    return g;
}

PT_DEV float4 sampleTrilinear(const DeviceScene &s, const DevTexture &t, uint32_t level, float frac, float u, float v)
{
    const float4 a = sampleBilinear(s, t, level, u, v);
    // single level, or a blend weight of exactly 0
    if (!(frac > 0.0f))
        return a;
    const float4 b = sampleBilinear(s, t, level + 1, u, v);
    return lerp4(a, b, frac);
}

// Inlined.  An out-of-line copy shrinks k_shade from 300 KB to 100 KB of SASS and removes the instruction-cache
// stalls, but the calls cost more than that saves (measured on the B200: shade 46.4 ms out of line vs 41.6 ms
// inlined, 32 spp of the chess scene).
static __device__ __forceinline__ float4 textureGrad(const DeviceScene &s, uint32_t slot, float u, float v, float4 deriv)
{
    const DevTexture &t = s.textures[slot];
    const GradFootprint g = gradFootprint(t, deriv, s.maxAnisotropy);
    if (g.taps == 1)
        return sampleTrilinear(s, t, g.level, g.frac, u, v);
    // the anisotropic taps: rare (grazing angles), kept out of the common path's registers
    float4 acc = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    const float n1 = (float)(g.taps + 1);
    for (uint32_t i = 1; i <= g.taps; i++)
    {
        const float o = (float)i / n1 - 0.5f;
        const float4 tap = sampleTrilinear(s, t, g.level, g.frac, u + o * g.du, v + o * g.dv);
        if (i == 1)
            acc = tap;
        else
            acc = make_float4(acc.x + tap.x, acc.y + tap.y, acc.z + tap.z, acc.w + tap.w);
    }
    const float n = (float)g.taps;
    return make_float4(acc.x / n, acc.y / n, acc.z / n, acc.w / n);
}

// texels textureGrad reads for this lookup (traversal statistics only)
PT_DEV uint32_t textureGradTexels(const DeviceScene &s, uint32_t slot, float4 deriv)
{
    const DevTexture &t = s.textures[slot];
    const GradFootprint g = gradFootprint(t, deriv, s.maxAnisotropy);
    auto texels = [&](uint32_t level) { return (max(1u, t.width >> level) == 1 && max(1u, t.height >> level) == 1) ? 1u : 4u; };
    return g.taps * (texels(g.level) + (g.frac > 0.0f ? texels(g.level + 1) : 0u));
}

} // namespace pt
