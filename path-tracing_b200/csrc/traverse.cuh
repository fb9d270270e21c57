// traverse.cuh — software traceRayEXT: BVH4 traversal + watertight ray/triangle test
// (Woop, Benthin, Wald, JCGT 2013) + the two any-hit shaders, for sm_100a.
//
// Replaces the fixed-function TLAS->BLAS traversal behind PT/Shaders/raygen.rgen:31,68.
// Closest-hit contract: nearest accepted hit with tmin < t < tmax; equal t resolved towards the
// smaller flattened triangle id (deterministic, BVH-independent).  Non-opaque candidates run the
// alpha test of anyhit.rahit:36-65 (closest) / occlusionAnyhit.rahit:35-54 (shadow).
#pragma once
#include "scene.cuh"

namespace pt
{

#define PT_STACK_SIZE 96 // >= 3 entries per level of the wide BVH + 1 (depths seen: 14-21); an overflow fails the call
// The stack lives in local memory.  Its first entries in SHARED memory instead were measured on the B200 (chess /
// street / atrium, 8 blocks per SM): 8 entries = no change, 16 entries = 1-3 % SLOWER, 24 entries = 8 % slower in
// k_extend — the hot top of a local-memory stack already sits in L1, and the shared-memory carve-out takes that L1
// away from the BVH nodes.

// the node phase of a warp goes on while more than this many lanes still look for their first leaf
// (0 = until every lane has one; lanes cut short idle through the triangle phase)
#ifndef PT_NODE_LOOP_LANES
#define PT_NODE_LOOP_LANES 4 // measured on chess: 0 -> 4 = k_extend -1.5 %, k_shadow -6 %; 8 = no further gain
#endif
// Entries a traversal could not push because its stack (PT_STACK_SIZE entries) was full.  A dropped entry is a lost
// sub-tree, i.e. possibly a missed hit: the host reads this counter after every call and FAILS the call when it is
// non-zero (checkStackOverflow).  The build also reports the depth of the wide BVH (pt_stats::bvh_max_depth).
static __device__ unsigned int g_stackOverflows;

PT_DEV void prefetchL1(const void *p) { asm volatile("prefetch.global.L1 [%0];" ::"l"(p)); }

struct Hit
{
    uint32_t tri; // leaf-order triangle index, 0xffffffff = miss
    float t, b1, b2;
};

// decal record of anyhit.rahit:54-62
struct Decal
{
    float dist; // -1 = none
    float r, g, b, a;
};

struct TraversalStats
{
    uint32_t boxTests, triTests, alphaTests;
};

// diagnostics of the persistent traversal (stats runs only): where the tail of a launch comes from
struct TailStats
{
    unsigned long long *visitHist; // [8]
    unsigned long long *warpIters, *warpDrainIters, *maxWarpDrainIters;
};

struct RaySetup
{
    vec3 org;
    float idx, idy, idz; // 1 / dir
    float Sx, Sy, Sz;
    int kx, ky, kz;
    // non-zero when the ray enters the slab of that axis through its hi plane: chosen by the SIGN BIT of the
    // direction (so that -0 pairs with idx = -inf)
    int nearX, nearY, nearZ;
};

// v[k] as two selects (FSEL) on predicates that depend on the ray only.  Written as the nested
// k == 0 ? v.x : (k == 1 ? v.y : v.z), ptxas made every one of the watertight test's nine components a divergent
// branch (BSSY / BRA / BSYNC; 7.6 % of k_extend's instructions at 14 of 32 lanes).
PT_DEV float comp(vec3 v, int k)
{
    const float yz = k == 1 ? v.y : v.z;
    return k == 0 ? v.x : yz;
}

PT_DEV RaySetup setupRay(vec3 o, vec3 d)
{
    RaySetup r;
    r.org = o;
    r.idx = 1.0f / d.x;
    r.idy = 1.0f / d.y;
    r.idz = 1.0f / d.z;
    const float ax = fabsf(d.x), ay = fabsf(d.y), az = fabsf(d.z);
    r.kz = (ax > ay) ? ((ax > az) ? 0 : 2) : ((ay > az) ? 1 : 2);
    r.kx = r.kz == 2 ? 0 : r.kz + 1;
    r.ky = r.kx == 2 ? 0 : r.kx + 1;
    const float dz = comp(d, r.kz);
    if (dz < 0.0f)
    {
        const int t = r.kx;
        r.kx = r.ky;
        r.ky = t;
    }
    r.Sx = comp(d, r.kx) / dz;
    r.Sy = comp(d, r.ky) / dz;
    r.Sz = 1.0f / dz;
    r.nearX = __float_as_int(d.x) < 0 ? 3 : 0;
    r.nearY = __float_as_int(d.y) < 0 ? 3 : 0;
    r.nearZ = __float_as_int(d.z) < 0 ? 3 : 0;
    return r;
}

// Returns true with (t, b1, b2) if the line hits the triangle; the caller checks the t range.
PT_DEV bool intersectTriangle(const RaySetup &r, vec3 p0, vec3 p1, vec3 p2, float &t, float &b1, float &b2)
{
    const vec3 A = p0 - r.org, B = p1 - r.org, C = p2 - r.org;
    const float Akz = comp(A, r.kz), Bkz = comp(B, r.kz), Ckz = comp(C, r.kz);
    const float Ax = comp(A, r.kx) - r.Sx * Akz, Ay = comp(A, r.ky) - r.Sy * Akz;
    const float Bx = comp(B, r.kx) - r.Sx * Bkz, By = comp(B, r.ky) - r.Sy * Bkz;
    const float Cx = comp(C, r.kx) - r.Sx * Ckz, Cy = comp(C, r.ky) - r.Sy * Ckz;
    // The edge functions must NOT be contracted into FMAs: watertightness relies on the two
    // triangles sharing an edge computing exactly opposite values (a*b - c*d with both products
    // rounded), which fma(a, b, -(c*d)) breaks — it also makes zero-area triangles "hit".
    float U = __fsub_rn(__fmul_rn(Cx, By), __fmul_rn(Cy, Bx));
    float V = __fsub_rn(__fmul_rn(Ax, Cy), __fmul_rn(Ay, Cx));
    float W = __fsub_rn(__fmul_rn(Bx, Ay), __fmul_rn(By, Ax));
    if (U == 0.0f || V == 0.0f || W == 0.0f)
    {
        U = (float)((double)Cx * (double)By - (double)Cy * (double)Bx);
        V = (float)((double)Ax * (double)Cy - (double)Ay * (double)Cx);
        W = (float)((double)Bx * (double)Ay - (double)By * (double)Ax);
    }
    if ((U < 0.0f || V < 0.0f || W < 0.0f) && (U > 0.0f || V > 0.0f || W > 0.0f))
        return false;
    const float det = U + V + W;
    if (det == 0.0f)
        return false;
    const float T = U * (r.Sz * Akz) + V * (r.Sz * Bkz) + W * (r.Sz * Ckz);
    const float rcpDet = 1.0f / det;
    t = T * rcpDet;
    b1 = V * rcpDet;
    b2 = W * rcpDet;
    return true;
}

// colour texture x colour factor at a candidate hit (anyhit.rahit:36-51, occlusionAnyhit.rahit:35-50), in two
// steps: the alpha channel decides (>= 0.5 accepts a closest-hit candidate, >= 1 an occluder), and only an IGNORED
// closest-hit candidate that is the nearest one so far needs the colour (the decal record).  Same texels, same
// weights, same per-channel arithmetic as sampleBilinear(level 0) — the three colour channels are simply evaluated
// later, or never: 12 of the 16 dependent table look-ups and 27 of the 36 interpolation operations of a test.
struct AnyHitSample
{
    float4 factor;
    float4 full;                // the whole colour where the two-step path does not apply (float / 1x1 textures)
    uint32_t t00, t10, t01, t11; // RGBA8 texels of the footprint
    float fx, fy;
    uint32_t lutOffset; // 256 = sRGB decode of the colour channels
    bool whole;
};

PT_DEV float anyHitAlpha(const DeviceScene &s, uint32_t shadeIndex, uint32_t materialId, float b1, float b2, AnyHitSample &a)
{
    const TriShade &ts = s.triShade[shadeIndex];
    const float4 a6 = __ldg(&ts.a[6]), a7 = __ldg(&ts.a[7]), a8 = __ldg(&ts.a[8]);
    const float b0 = 1.0f - b1 - b2;
    float u = a6.w * b0 + a7.y * b1 + a7.w * b2;
    float v = a7.x * b0 + a7.z * b1 + a8.x * b2;
    const uint32_t type = materialId & 0xffu, index = materialId >> 8;
    a.whole = true;
    if (type > 2)
    {
        a.full = make_float4(1.0f, 0.0f, 0.0f, 1.0f); // getColorFactor default, texture 0 is white
        return 1.0f;
    }
    const MaterialRaw *m = (type == 0 ? s.materials[0] : type == 1 ? s.materials[1] : s.materials[2]) + index;
    a.factor = __ldg(&m->q[1]); // vec4 Color sits at byte 16 in all three structs
    // ColorIdx: MR byte 80 (q[5].x); SG / Phong byte 76 (q[4].w)
    const uint32_t colorIdx =
        type == 0 ? __float_as_uint(__ldg(&m->q[5]).x) : __float_as_uint(__ldg(&m->q[4]).w);
    const DevTexture &t = s.textures[colorIdx];
    const uint32_t lw = t.width, lh = t.height, flags = t.flags;
    if ((flags & PT_TEX_FLAG_FLOAT) || (lw == 1 && lh == 1))
    {
        const float4 c = textureLod0(s, t, u, v);
        a.full = make_float4(c.x * a.factor.x, c.y * a.factor.y, c.z * a.factor.z, c.w * a.factor.w);
        return a.full.w;
    }
    a.whole = false;
    a.lutOffset = (flags & PT_TEX_FLAG_SRGB) ? 256u : 0u;
    // sampleBilinear(level 0): repeat wrap, texel centres at half integers
    u = isfinite(u) ? u : 0.0f;
    v = isfinite(v) ? v : 0.0f;
    u = u - floorf(u);
    v = v - floorf(v);
    const float x = u * (float)lw - 0.5f, y = v * (float)lh - 0.5f;
    const float fx0 = floorf(x), fy0 = floorf(y);
    a.fx = x - fx0, a.fy = y - fy0;
    const int W = (int)lw, H = (int)lh;
    const int ix = (int)fx0, iy = (int)fy0;
    const int x0 = ix < 0 ? W - 1 : ix, x1 = x0 + 1 == W ? 0 : x0 + 1;
    const int y0 = iy < 0 ? H - 1 : iy, y1 = y0 + 1 == H ? 0 : y0 + 1;
    const uint32_t *texels = reinterpret_cast<const uint32_t *>(t.base) + t.levelOffset[0];
    a.t00 = __ldg(texels + (size_t)y0 * lw + x0), a.t10 = __ldg(texels + (size_t)y0 * lw + x1);
    a.t01 = __ldg(texels + (size_t)y1 * lw + x0), a.t11 = __ldg(texels + (size_t)y1 * lw + x1);
    // alpha is never sRGB-encoded: table entries [0, 255]
    const float a00 = __ldg(s.lut + (a.t00 >> 24)), a10 = __ldg(s.lut + (a.t10 >> 24));
    const float a01 = __ldg(s.lut + (a.t01 >> 24)), a11 = __ldg(s.lut + (a.t11 >> 24));
    const float gx = 1.0f - a.fx, gy = 1.0f - a.fy;
    const float top = a00 * gx + a10 * a.fx, bottom = a01 * gx + a11 * a.fx;
    return (top * gy + bottom * a.fy) * a.factor.w;
}

// the colour channels of the sample anyHitAlpha looked at (x factor)
PT_DEV vec3 anyHitRgb(const DeviceScene &s, const AnyHitSample &a)
{
    if (a.whole)
        return V3(a.full);
    const float *lut = s.lut + a.lutOffset;
    const float gx = 1.0f - a.fx, gy = 1.0f - a.fy;
    float c[3];
#pragma unroll
    for (int k = 0; k < 3; k++)
    {
        const float c00 = __ldg(lut + ((a.t00 >> (8 * k)) & 0xffu)), c10 = __ldg(lut + ((a.t10 >> (8 * k)) & 0xffu));
        const float c01 = __ldg(lut + ((a.t01 >> (8 * k)) & 0xffu)), c11 = __ldg(lut + ((a.t11 >> (8 * k)) & 0xffu));
        const float top = c00 * gx + c10 * a.fx, bottom = c01 * gx + c11 * a.fx;
        c[k] = top * gy + bottom * a.fy;
    }
    return V3(c[0] * a.factor.x, c[1] * a.factor.y, c[2] * a.factor.z);
}

// One BVH4 node: tests the four child boxes, returns entry distances (INF if missed / empty).
// The entry / exit plane words of every slab are picked once per node by the ray's direction signs,
// so a box costs six byte conversions, six FMAs and two four-input max / min.
PT_DEV void intersectNode(const BvhNode *__restrict__ node, const RaySetup &r, float tmin, float tmax, float d[4],
                          int c[4])
{
    const uint4 *q = reinterpret_cast<const uint4 *>(node);
    const uint4 w0 = __ldg(q), w1 = __ldg(q + 1), w2 = __ldg(q + 2);
    const int4 ch = __ldg(&node->child);
    c[0] = ch.x, c[1] = ch.y, c[2] = ch.z, c[3] = ch.w;
    // plane distance = (origin + k * step - org) * idir = k * (step * idir) + (origin - org) * idir: one FMA per
    // plane.  A non-finite product (axis-parallel ray) yields NaN, which fminf / fmaxf drop: the axis then
    // does not constrain the box — conservative.
    const float ax = __uint_as_float(w0.w) * r.idx, ay = __uint_as_float(w1.x) * r.idy, az = __uint_as_float(w1.y) * r.idz;
    const float bx = (__uint_as_float(w0.x) - r.org.x) * r.idx, by = (__uint_as_float(w0.y) - r.org.y) * r.idy;
    const float bz = (__uint_as_float(w0.z) - r.org.z) * r.idz;
    // The rounding of fmaf(k, a, b) is ABSOLUTE, a few ulp of |b| + 255 |a| (the distances of the node's planes), not of the
    // result: for a ray that starts near a surface inside a large node (every continuation ray) it exceeds any relative
    // slack, and a box whose face holds the edge or vertex the ray crosses was culled — rays leaked through closed meshes,
    // and ties at shared vertices depended on the visiting order.  Entry planes therefore move 4 units of roundoff of their
    // axis' terms closer, exit planes as much farther, plus the same of the dominant axis kz, which bounds the rounding of
    // the t of a triangle inside the node.  (A zero direction component makes its axis NaN, which the min / max drop.)
    const float ex = fmaf(255.0f, fabsf(ax), fabsf(bx)), ey = fmaf(255.0f, fabsf(ay), fabsf(by));
    const float ez = fmaf(255.0f, fabsf(az), fabsf(bz));
    const float kErr = 2.3841858e-7f; // 4 * 2^-24
    const float eKz = kErr * comp(V3(ex, ey, ez), r.kz);
    const float sx = fmaf(kErr, ex, eKz), sy = fmaf(kErr, ey, eKz), sz = fmaf(kErr, ez, eKz);
    const float bnx = bx - sx, bfx = bx + sx, bny = by - sy, bfy = by + sy, bnz = bz - sz, bfz = bz + sz;
    // entry / exit planes by the sign of the direction
    const uint32_t nxw = r.nearX ? w2.y : w1.z, fxw = r.nearX ? w1.z : w2.y;
    const uint32_t nyw = r.nearY ? w2.z : w1.w, fyw = r.nearY ? w1.w : w2.z;
    const uint32_t nzw = r.nearZ ? w2.w : w2.x, fzw = r.nearZ ? w2.x : w2.w;
#pragma unroll
    for (int i = 0; i < 4; i++)
    {
        const float tnx = fmaf((float)((nxw >> (8 * i)) & 0xffu), ax, bnx), tfx = fmaf((float)((fxw >> (8 * i)) & 0xffu), ax, bfx);
        const float tny = fmaf((float)((nyw >> (8 * i)) & 0xffu), ay, bny), tfy = fmaf((float)((fyw >> (8 * i)) & 0xffu), ay, bfy);
        const float tnz = fmaf((float)((nzw >> (8 * i)) & 0xffu), az, bnz), tfz = fmaf((float)((fzw >> (8 * i)) & 0xffu), az, bfz);
        const float t0 = fmaxf(fmaxf(tnx, tny), fmaxf(tnz, tmin));
        const float t1 = fminf(fminf(tfx, tfy), fminf(tfz, tmax));
        // the relative slack absorbs the rounding of t0 and t1 themselves
        d[i] = (c[i] != PT_CHILD_EMPTY && t0 <= t1 * 1.0000008f) ? t0 : INFINITY;
    }
}

// distances by min / max, references by one compare and two selects (an if-swap compiled to eight moves);
// the distances are never NaN, so min / max order them as the compare does
#define PT_CSWAP(i, j)                                                                                                \
    {                                                                                                                 \
        const bool sw = d[j] < d[i];                                                                                  \
        const int ci = sw ? c[j] : c[i], cj = sw ? c[i] : c[j];                                                       \
        const float di = fminf(d[i], d[j]), dj = fmaxf(d[i], d[j]);                                                   \
        d[i] = di, d[j] = dj, c[i] = ci, c[j] = cj;                                                                   \
    }

// cur value "take the next entry off the stack": popping is a step of the state machine of its own
// (popStep), executed by all lanes of a warp together, instead of a loop inside whichever lane
// runs dry — that loop ran with 4 of 32 lanes active and a dependent local-memory load per trip.
#define PT_CHILD_POP 0x7ffffffe

// Per-lane traversal state machine.  `cur` is the next thing to do: an internal node (>= 0), a
// leaf (< 0), PT_CHILD_POP = fetch the next stack entry, or PT_CHILD_EMPTY = finished.  The kernels drive it either as a plain per-thread
// loop (traverse(), standalone queries) or warp-synchronously with dynamic ray fetch (wavefront).
//   CLOSEST = true : nearest hit (+ decal record if ALPHA)
//   CLOSEST = false: any hit in (tmin, tmax) with alpha >= 1 -> hit.tri != miss
//   CULL = true    : gl_RayFlagsCullBackFacingTrianglesEXT (debug pipeline only): back-facing triangles are no
//                    candidates at all.  Vulkan decides the facing in OBJECT space: front = the vertices appear
//                    clockwise from the ray origin, i.e. dot((v1 - v0) x (v2 - v0), d) < 0 there; a mirroring
//                    instance transform reverses the world-space winding (PT_TRI_FLAG_MIRRORED).
template <bool CLOSEST, bool ALPHA, bool STATS, bool CULL = false> struct Traverser
{
    vec3 cullDir; // world ray direction (CULL only)
    static constexpr bool kClosest = CLOSEST, kAlpha = ALPHA, kStats = STATS;
    RaySetup r;
    float tmin, tmax, best;
    uint32_t bestFlat;
    Hit hit;
    Decal decal;
    TraversalStats st;
    uint32_t visits; // nodes visited by the current ray (diagnostics)
    int cur;
    int leaf; // postponed leaf (speculative traversal), PT_CHILD_EMPTY = none
    int sp;
    // (entry distance bits << 32) | node reference.  The array lives OUTSIDE the struct (a
    // dynamically indexed member would drag every scalar field into local memory with it).
    unsigned long long *stack;

    PT_DEV bool finished() const { return cur == PT_CHILD_EMPTY && leaf == PT_CHILD_EMPTY; }
    PT_DEV bool hasLeaf() const { return leaf != PT_CHILD_EMPTY; }
    PT_DEV bool atInternal() const { return (unsigned)cur < (unsigned)PT_CHILD_POP; }
    PT_DEV bool needsPop() const { return cur == PT_CHILD_POP; }

    PT_DEV void begin(const DeviceScene &s, vec3 org, vec3 dir, float tmin_, float tmax_)
    {
        tmin = tmin_;
        tmax = tmax_;
        best = tmax_;
        bestFlat = 0xffffffffu;
        hit.tri = 0xffffffffu;
        hit.t = tmax_;
        hit.b1 = hit.b2 = 0.0f;
        if (ALPHA)
            decal.dist = -1.0f;
        sp = 0;
        visits = 0;
        leaf = PT_CHILD_EMPTY;
        cur = 0; // the root is always an internal node
        // A ray with a non-finite component or a zero direction cannot hit anything (every triangle
        // test evaluates to NaN), but NaN also defeats box culling, so it would walk the WHOLE tree.
        // Such rays exist by design: refract() returns 0 on total internal reflection and
        // normalize(0) is NaN (SURVEY Q12); the sample is then restarted (Q7).  Miss immediately.
        const float sum = org.x + org.y + org.z + dir.x + dir.y + dir.z;
        if (s.triCount == 0 || !isfinite(sum) || (dir.x == 0.0f && dir.y == 0.0f && dir.z == 0.0f))
            cur = PT_CHILD_EMPTY;
        r = setupRay(org, dir);
    }

    // One stack entry, if the lane asked for it: sub-trees that start beyond the current best are
    // dropped (ties are kept) and the lane asks again.
    PT_DEV void popStep()
    {
        if (cur != PT_CHILD_POP)
            return;
        if (sp == 0)
        {
            cur = PT_CHILD_EMPTY;
            return;
        }
        const unsigned long long e = take();
        if (!CLOSEST || __uint_as_float((uint32_t)(e >> 32)) <= best)
            cur = (int)(uint32_t)e;
    }

    // removes and returns the top entry (sp > 0)
    PT_DEV unsigned long long take()
    {
        --sp;
        return stack[sp];
    }

    PT_DEV void push(int node, float dist)
    {
        const unsigned long long e = ((unsigned long long)__float_as_uint(dist) << 32) | (uint32_t)node;
        if (sp < PT_STACK_SIZE)
        {
            stack[sp] = e;
            sp++;
        }
        else
            atomicAdd(&g_stackOverflows, 1u);
    }

    // cur is an internal node: test its children, descend into the nearest, push the others
    PT_DEV void nodeStep(const DeviceScene &s)
    {
        float d[4];
        int c[4];
        intersectNode(s.nodes + cur, r, tmin, best, d, c);
        if (STATS)
        {
            st.boxTests += 4;
            visits++;
        }
        // sorting network, ascending by distance (missed children carry INF).  Occlusion rays are sorted too:
        // taking the hit children in stored order was measured k_shadow -3 % on chess, -1 % dragon, +8 % street —
        // near-first order finds occluders sooner.
        PT_CSWAP(0, 1)
        PT_CSWAP(2, 3)
        PT_CSWAP(0, 2)
        PT_CSWAP(1, 3)
        PT_CSWAP(1, 2)
        if (d[0] == INFINITY)
        {
            cur = PT_CHILD_POP;
            return;
        }
        cur = c[0];
        // the hit children are d[0 .. m]: the rest goes on the stack farthest first, as predicated stores below one
        // bound check (three conditional pushes were three branches with a bound check each)
        const bool h1 = d[1] != INFINITY, h2 = d[2] != INFINITY, h3 = d[3] != INFINITY;
        const int m = (int)h1 + (int)h2 + (int)h3;
        if (sp + m <= PT_STACK_SIZE)
        {
            unsigned long long *top = stack + sp + m; // one past the new top
            if (h1)
                top[-1] = ((unsigned long long)__float_as_uint(d[1]) << 32) | (uint32_t)c[1];
            if (h2)
                top[-2] = ((unsigned long long)__float_as_uint(d[2]) << 32) | (uint32_t)c[2];
            if (h3)
                top[-3] = ((unsigned long long)__float_as_uint(d[3]) << 32) | (uint32_t)c[3];
            sp += m;
            return;
        }
        // push the rest, farthest first
        if (d[3] != INFINITY)
            push(c[3], d[3]);
        if (d[2] != INFINITY)
            push(c[2], d[2]);
        if (d[1] != INFINITY)
            push(c[1], d[1]);
    }

    // result of another lane that traversed part of this ray's tree (straggler splitting)
    PT_DEV void merge(uint32_t tri, float t, float b1, float b2, uint32_t flat)
    {
        if (tri == 0xffffffffu)
            return;
        if (CLOSEST)
        {
            if (!(t < best || (t == best && flat < bestFlat)))
                return;
            best = t;
            bestFlat = flat;
        }
        else
        {
            cur = leaf = PT_CHILD_EMPTY; // occluded: nothing left to do
            sp = 0;
        }
        hit.tri = tri;
        hit.t = t;
        hit.b1 = b1;
        hit.b2 = b2;
    }

    // speculative traversal (Aila & Laine 2009): the first leaf found is set aside and the lane keeps
    // descending, so that the lanes of a warp reach the triangle tests together
    PT_DEV void postponeLeaf(const float4 *sPrefetchTri)
    {
        if (cur < 0 && leaf == PT_CHILD_EMPTY)
        {
            leaf = cur;
            prefetchL1(sPrefetchTri + 3 * (size_t)(((uint32_t)~cur) >> 2)); // the leaf's first triangle, into L1
            cur = PT_CHILD_POP;
        }
    }

    // tests the triangles of the postponed leaf (and, if ALPHA, of a second leaf waiting in cur)
    PT_DEV void leafStep(const DeviceScene &s)
    {
        while (leaf != PT_CHILD_EMPTY)
        {
            const uint32_t code = (uint32_t)~leaf;
            const uint32_t first = code >> 2, count = (code & 3u) + 1;
            leaf = PT_CHILD_EMPTY;
            for (uint32_t i = 0; i < count; i++)
            {
                const uint32_t tri = first + i;
                const float4 q0 = __ldg(s.triPos + 3 * (size_t)tri);
                const float4 q1 = __ldg(s.triPos + 3 * (size_t)tri + 1);
                const float4 q2 = __ldg(s.triPos + 3 * (size_t)tri + 2);
                if (STATS)
                    st.triTests++;
                float t, b1, b2;
                if (!intersectTriangle(r, V3(q0), V3(q1), V3(q2), t, b1, b2))
                    continue;
                if (!(t > tmin))
                    continue;
                const uint32_t flat = __float_as_uint(q0.w);
                if (CULL)
                {
                    const vec3 n = cross(V3(q1) - V3(q0), V3(q2) - V3(q0));
                    float facing = dot(n, cullDir);
                    if (__float_as_uint(q1.w) & PT_TRI_FLAG_MIRRORED)
                        facing = -facing;
                    if (!(facing < 0.0f))
                        continue; // back-facing (or edge-on)
                }
                if (CLOSEST)
                {
                    if (!(t < best || (t == best && flat < bestFlat)))
                        continue;
                }
                else if (!(t < tmax))
                    continue;
                if (ALPHA && !(__float_as_uint(q1.w) & PT_TRI_FLAG_OPAQUE))
                {
                    if (STATS)
                        st.alphaTests++;
                    AnyHitSample ah;
                    const float alpha = anyHitAlpha(s, __float_as_uint(q0.w), __float_as_uint(q2.w), b1, b2, ah);
                    if (CLOSEST)
                    {
                        if (alpha < 0.5f)
                        {
                            if (decal.dist == -1.0f || t < decal.dist)
                            {
                                const vec3 rgb = anyHitRgb(s, ah);
                                decal.r = rgb.x, decal.g = rgb.y, decal.b = rgb.z, decal.a = alpha;
                                decal.dist = t;
                            }
                            continue; // ignoreIntersectionEXT
                        }
                    }
                    else if (alpha < 1.0f)
                        continue;
                }
                hit.tri = tri;
                hit.t = t;
                hit.b1 = b1;
                hit.b2 = b2;
                if (!CLOSEST)
                {
                    cur = leaf = PT_CHILD_EMPTY; // gl_RayFlagsTerminateOnFirstHitEXT
                    sp = 0;
                    return;
                }
                best = t;
                bestFlat = flat;
            }
            // a second leaf found while this one was postponed (scenes with alpha-tested geometry visit many
            // leaves per ray — 20 in the atrium — and are 2.5 % faster chaining them; the others are 2.3-2.5 %
            // faster leaving it to the next round of the warp)
            if (ALPHA && cur < 0)
            {
                leaf = cur;
                cur = PT_CHILD_POP;
            }
        }
    }
};

// plain per-thread traversal (standalone queries)
template <bool CLOSEST, bool ALPHA, bool STATS, bool CULL = false>
PT_DEV void traverse(const DeviceScene &s, vec3 org, vec3 dir, float tmin, float tmax, Hit &hit, Decal &decal,
                     TraversalStats &st)
{
    unsigned long long stack[PT_STACK_SIZE];
    Traverser<CLOSEST, ALPHA, STATS, CULL> tr;
    tr.stack = stack;
    tr.cullDir = dir;
    tr.st = st;
    tr.begin(s, org, dir, tmin, tmax);
    while (!tr.finished())
    {
        while (tr.atInternal() || tr.needsPop())
        {
            if (tr.atInternal())
                tr.nodeStep(s);
            tr.popStep();
        }
        tr.postponeLeaf(s.triPos);
        tr.popStep();
        tr.leafStep(s);
    }
    hit = tr.hit;
    decal = tr.decal;
    st = tr.st;
}

// ---------------------------------------------------------------------------------------------
// Warp-synchronous traversal with dynamic ray fetch (Aila & Laine 2009, persistent warps).
//
// Every warp of a persistent grid keeps 32 traversal state machines.  Rays differ wildly in
// length; instead of letting finished lanes idle until the longest ray of the warp is done, the
// warp refills its idle lanes from the ray queue as soon as fewer than PT_REFILL_LANES lanes are
// still traversing.  Queue positions are handed out to warps in chunks of PT_FETCH_CHUNK through
// one atomic per chunk; inside a chunk lanes take positions by ballot arithmetic.
//
//   loadSlot(i)        : issue the load of queue entry i (the slot index, possibly with flag bits)
//   loadRay(entry)     : issue the loads of that entry's ray, return them as a RayPacket (k_extend also
//                        regenerates ended paths here; slot 0xffffffff = no ray)
//   commit(tr, slot)   : ray finished — write the result
//
// Two details matter as much as the refill itself:
//   * ray PREFETCH: a refill needs queue -> slot -> ray, two dependent DRAM round trips during which
//     the whole warp would stall.  The warp therefore keeps the next 32 rays of its chunk in
//     registers (lane L holds buffered ray L); a refill is a handful of shuffles, and the loads
//     for the following 32 rays are issued right away, to complete behind the traversal work
//     (two stages: the slot indices of batch k+2 are requested together with the rays of batch k+1,
//     so neither of the two dependent loads is ever waited for).
//   * DEFERRED commit: finished lanes keep their result until the next refill point, where all of
//     them push to the hit / done queues together — one aggregated atomic per queue and refill
//     instead of one per lane (same-address atomics are serialised by the L2).
//   * STRAGGLER SPLITTING: once the queue is empty a warp only drains, and the kernel lasts as
//     long as its longest ray (a ray grazing a tessellated floor visits thousands of nodes while
//     the rest of the GPU idles).  In drain mode idle lanes therefore take sub-trees off the
//     deepest stack of the warp: the donor pops an entry, the helper copies the ray and traverses
//     that sub-tree, and its result is merged into the owner's with the same (t, triangle id)
//     order the serial traversal uses — the answer is identical, the tail up to 32x shorter.
// ---------------------------------------------------------------------------------------------
#ifndef PT_FETCH_CHUNK
#define PT_FETCH_CHUNK 32u
#endif
#ifndef PT_REFILL_LANES
#define PT_REFILL_LANES 20
#endif

struct RayPacket
{
    uint32_t slot;
    float ox, oy, oz, dx, dy, dz, tmax;
};

template <class TR, class LoadSlot, class LoadRay, class Commit>
PT_DEV void tracePersistent(const DeviceScene &s, uint32_t n, uint32_t *workCounter, TR &tr, float tmin,
                            LoadSlot loadSlot, LoadRay loadRay, Commit commit, TailStats tail)
{
    uint32_t dbgIters = 0, dbgDrainIters = 0;
    auto countVisits = [&](uint32_t v) {
        if (TR::kStats)
        {
            const int bin = v < 16 ? 0 : min(7, 28 - __clz(v));
            atomicAdd(tail.visitHist + bin, 1ull);
        }
    };
    const unsigned FULL = 0xffffffffu;
    const unsigned lane = threadIdx.x & 31u;
    const unsigned ltMask = (1u << lane) - 1u;
    uint32_t wBase = 0, wEnd = 0; // warp-uniform: the not yet buffered rest of the warp's chunk
    bool exhausted = false;       // warp-uniform: the queue has no more chunks
    uint32_t pfPos = 0, pfCount = 0; // warp-uniform: lanes [pfPos, pfCount) hold buffered rays
    RayPacket pf = {};
    bool haveRay = false, pending = false;
    uint32_t slot = 0;
    unsigned owner = lane; // lane whose ray this lane works on (differs only for drain-mode helpers)
    tr.cur = tr.leaf = PT_CHILD_EMPTY;

    uint32_t nxCount = 0; // warp-uniform: lanes [0, nxCount) hold the slot indices of the batch after the buffer
    uint32_t nxSlot = 0;
    // (both stages are force-inlined: as calls they forced a local-memory copy of the kernel parameter block, DESIGN.md §3)
    // stage 1: request the slot indices of the next batch of the warp's chunk
    auto prefetchSlots = [&]() __attribute__((always_inline)) {
        nxCount = 0;
        if (exhausted)
            return;
        if (wBase == wEnd)
        {
            uint32_t b = 0;
            if (lane == 0)
                b = atomicAdd(workCounter, PT_FETCH_CHUNK);
            b = __shfl_sync(FULL, b, 0);
            if (b >= n)
            {
                exhausted = true;
                return;
            }
            wBase = b;
            wEnd = min(b + PT_FETCH_CHUNK, n);
        }
        nxCount = min(32u, wEnd - wBase);
        if (lane < nxCount)
            nxSlot = loadSlot(wBase + lane);
        wBase += nxCount;
    };
    // stage 2: request the rays of the batch whose slot indices arrived meanwhile, then stage 1 again
    auto prefetch = [&]() __attribute__((always_inline)) {
        pfPos = 0;
        pfCount = nxCount;
        if (lane < nxCount)
            pf = loadRay(nxSlot);
        prefetchSlots();
    };
    prefetchSlots();
    prefetch();

    for (;;)
    {
        // ---- results of the lanes that finished since the last refill -------------------------------
        if (pending)
            commit(tr, slot);
        pending = false;
        // ---- refill idle lanes from the register buffer ----------------------------------------
        unsigned idle = __ballot_sync(FULL, !haveRay);
        while (idle != 0 && pfPos < pfCount)
        {
            const uint32_t take = min((uint32_t)__popc(idle), pfCount - pfPos);
            const uint32_t rank = __popc(idle & ltMask);
            const int src = (int)((pfPos + rank) & 31u);
            RayPacket p;
            p.slot = __shfl_sync(FULL, pf.slot, src);
            p.ox = __shfl_sync(FULL, pf.ox, src);
            p.oy = __shfl_sync(FULL, pf.oy, src);
            p.oz = __shfl_sync(FULL, pf.oz, src);
            p.dx = __shfl_sync(FULL, pf.dx, src);
            p.dy = __shfl_sync(FULL, pf.dy, src);
            p.dz = __shfl_sync(FULL, pf.dz, src);
            p.tmax = __shfl_sync(FULL, pf.tmax, src);
            // (a packet with slot 0xffffffff carries no ray: the lane stays idle and is offered the next one)
            if (!haveRay && rank < take && p.slot != 0xffffffffu)
            {
                slot = p.slot;
                owner = lane;
                tr.begin(s, V3(p.ox, p.oy, p.oz), V3(p.dx, p.dy, p.dz), tmin, p.tmax);
                haveRay = true;
            }
            pfPos += take;
            if (pfPos == pfCount && nxCount != 0)
                prefetch(); // loads complete behind the traversal below
            idle = __ballot_sync(FULL, !haveRay);
        }
        if (idle == FULL)
        {
            if (TR::kStats && lane == 0)
            {
                atomicAdd(tail.warpIters, (unsigned long long)dbgIters);
                atomicAdd(tail.warpDrainIters, (unsigned long long)dbgDrainIters);
                atomicMax(tail.maxWarpDrainIters, (unsigned long long)dbgDrainIters);
            }
            return; // nothing left anywhere
        }
        // ---- traverse until too many lanes have finished -----------------------------------------
        const bool drain = pfPos == pfCount; // warp-uniform: nothing left to refill with
        for (;;)
        {
            // internal nodes, until every lane either holds a leaf or has nothing left to descend into;
            // lanes that already hold a leaf keep traversing speculatively meanwhile
            do
            {
                if (tr.atInternal())
                    tr.nodeStep(s);
                tr.postponeLeaf(s.triPos);
                tr.popStep();
            } while (__popc(__ballot_sync(FULL, (tr.atInternal() || tr.needsPop()) && !tr.hasLeaf())) > PT_NODE_LOOP_LANES);
            tr.leafStep(s);
            if (!drain)
            {
                if (TR::kStats)
                    dbgIters++;
                if (haveRay && tr.finished())
                {
                    countVisits(tr.visits);
                    pending = true;
                    haveRay = false;
                }
                if (__popc(__ballot_sync(FULL, haveRay)) < PT_REFILL_LANES)
                    break;
                continue;
            }
            // ---- drain mode -----------------------------------------------------------------------
            if (TR::kStats)
            {
                dbgIters++;
                dbgDrainIters++;
            }
            // (1) helpers that are done hand their result to the owner lane
            unsigned hm = __ballot_sync(FULL, haveRay && owner != lane && tr.finished());
            while (hm != 0)
            {
                const int h = __ffs(hm) - 1;
                hm &= hm - 1;
                const unsigned o = __shfl_sync(FULL, owner, h);
                const uint32_t tri = __shfl_sync(FULL, tr.hit.tri, h);
                const float t = __shfl_sync(FULL, tr.hit.t, h);
                const float b1 = __shfl_sync(FULL, tr.hit.b1, h), b2 = __shfl_sync(FULL, tr.hit.b2, h);
                const uint32_t flat = __shfl_sync(FULL, tr.bestFlat, h);
                const float dd = __shfl_sync(FULL, tr.decal.dist, h), dr = __shfl_sync(FULL, tr.decal.r, h);
                const float dg = __shfl_sync(FULL, tr.decal.g, h), db = __shfl_sync(FULL, tr.decal.b, h);
                const float da = __shfl_sync(FULL, tr.decal.a, h);
                if ((int)lane == h)
                    haveRay = false;
                else if (haveRay && owner == o)
                {
                    // the owner takes the result; for occlusion rays every part of the ray stops on a hit
                    if (lane == o || !TR::kClosest)
                        tr.merge(tri, t, b1, b2, flat);
                    if (lane == o && TR::kAlpha && TR::kClosest && dd != -1.0f && (tr.decal.dist == -1.0f || dd < tr.decal.dist))
                    {
                        tr.decal.dist = dd;
                        tr.decal.r = dr, tr.decal.g = dg, tr.decal.b = db, tr.decal.a = da;
                    }
                }
            }
            // (2) owners whose ray is done in all its parts
            const unsigned group = __match_any_sync(FULL, haveRay ? owner : 32u + lane);
            if (haveRay && owner == lane && tr.finished() && group == (1u << lane))
            {
                countVisits(tr.visits);
                commit(tr, slot);
                haveRay = false;
            }
            // (3) idle lanes take sub-trees off the deepest stacks
            unsigned idleLanes = ~__ballot_sync(FULL, haveRay);
            if (idleLanes == FULL)
                break;
            while (idleLanes != 0)
            {
                const unsigned key = (haveRay && tr.sp >= 1) ? (((unsigned)tr.sp << 5) | lane) : 0u;
                const unsigned top = __reduce_max_sync(FULL, key);
                if (top == 0)
                    break;
                const int donor = (int)(top & 31u);
                const int helper = __ffs(idleLanes) - 1;
                idleLanes &= idleLanes - 1;
                unsigned long long e = 0;
                if ((int)lane == donor)
                    e = tr.take();
                e = __shfl_sync(FULL, e, donor);
                RaySetup r;
                r.org.x = __shfl_sync(FULL, tr.r.org.x, donor), r.org.y = __shfl_sync(FULL, tr.r.org.y, donor);
                r.org.z = __shfl_sync(FULL, tr.r.org.z, donor);
                r.idx = __shfl_sync(FULL, tr.r.idx, donor), r.idy = __shfl_sync(FULL, tr.r.idy, donor);
                r.idz = __shfl_sync(FULL, tr.r.idz, donor);
                r.Sx = __shfl_sync(FULL, tr.r.Sx, donor), r.Sy = __shfl_sync(FULL, tr.r.Sy, donor);
                r.Sz = __shfl_sync(FULL, tr.r.Sz, donor);
                r.kx = __shfl_sync(FULL, tr.r.kx, donor), r.ky = __shfl_sync(FULL, tr.r.ky, donor);
                r.kz = __shfl_sync(FULL, tr.r.kz, donor);
                r.nearX = __shfl_sync(FULL, tr.r.nearX, donor), r.nearY = __shfl_sync(FULL, tr.r.nearY, donor);
                r.nearZ = __shfl_sync(FULL, tr.r.nearZ, donor);
                const float dTmin = __shfl_sync(FULL, tr.tmin, donor), dTmax = __shfl_sync(FULL, tr.tmax, donor);
                const float dBest = __shfl_sync(FULL, tr.best, donor);
                const uint32_t dFlat = __shfl_sync(FULL, tr.bestFlat, donor);
                const uint32_t dSlot = __shfl_sync(FULL, slot, donor);
                const unsigned dOwner = __shfl_sync(FULL, owner, donor);
                if ((int)lane == helper)
                {
                    tr.r = r;
                    tr.tmin = dTmin;
                    tr.tmax = dTmax;
                    tr.best = dBest;
                    tr.bestFlat = dFlat;
                    tr.hit.tri = 0xffffffffu;
                    tr.hit.t = dTmax;
                    tr.hit.b1 = tr.hit.b2 = 0.0f;
                    tr.decal.dist = -1.0f;
                    tr.cur = (int)(uint32_t)e;
                    tr.leaf = PT_CHILD_EMPTY;
                    tr.sp = 0;
                    slot = dSlot;
                    owner = dOwner;
                    haveRay = true;
                }
            }
        }
    }
}

} // namespace pt
