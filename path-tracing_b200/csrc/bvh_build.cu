// bvh_build.cu — scene upload: transform baking, skinning and the GPU BVH build (textures: textures.cu).
//
// Replaces Renderer::UpdateSceneData's uploads (PT/Renderer/Renderer.cpp:251-399) and the
// driver-side acceleration-structure build requested by AccelerationStructure's constructor
// (PT/Renderer/AccelerationStructure.cpp:12-35, 64-165, 260-301) — the reference itself has no BVH
// code.  Pipeline, all on the GPU:
//   bake (instance x mesh transforms -> world-space triangles + shading records)
//   -> centroid bounds -> 63-bit Morton codes -> radix sort (CUB)
//   -> binary hierarchy: PLOC (Meister & Bittner 2018: repeated merging of mutually nearest clusters
//      inside a Morton-order window, nearest = smallest surface area of the union — the default) or
//      LBVH (Karras 2012, + bottom-up refit; tuning key "bvh_builder" = 0)
//   -> surface-area-guided collapse into 4-wide 128-byte nodes with <= 4-triangle leaves, which also
//      lays the triangles out in depth-first leaf order
//   -> gather triangles into leaf order.
#include "core_internal.h"

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include <algorithm>
#include <cmath>
#include <cstring>

namespace pt
{

namespace
{

// One (instance, mesh) pair of the flattened TLAS/BLAS hierarchy.
struct MeshInstance
{
    float P[12];  // P[j*4 + c]: world_j = p.x*P[j][0] + p.y*P[j][1] + p.z*P[j][2] + P[j][3]
    float N[9];   // normal matrix (inverse transpose of the linear part), row-major
    uint32_t triOffset, triCount;
    uint32_t vertexOffset, indexOffset;
    uint32_t vertexLength;       // vertices of the geometry: every index must be below it
    uint32_t instance, geometry; // gl_InstanceID, geometry index inside the model
    uint32_t materialId, flags;
};

struct Aabb
{
    float lo[3], hi[3];
};

__device__ __forceinline__ uint32_t floatFlip(float f)
{
    const uint32_t u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float floatUnflip(uint32_t u)
{
    return __uint_as_float((u & 0x80000000u) ? (u & 0x7fffffffu) : ~u);
}

// ---------------------------------------------------------------------------------------------
// bake
// ---------------------------------------------------------------------------------------------
__global__ void k_bake(const MeshInstance *__restrict__ mis, uint32_t miCount, const float *__restrict__ vertices,
                       const uint32_t *__restrict__ indices, uint32_t triCount, float4 *__restrict__ triPos,
                       TriShade *__restrict__ triShade, Aabb *__restrict__ boxes, uint32_t *__restrict__ sceneBounds,
                       uint32_t *__restrict__ badIndexCount)
{
    const uint32_t tri = blockIdx.x * blockDim.x + threadIdx.x;
    if (tri >= triCount)
        return;
    // binary search: last mesh instance with triOffset <= tri
    uint32_t lo = 0, hi = miCount - 1;
    while (lo < hi)
    {
        const uint32_t mid = (lo + hi + 1) >> 1;
        if (mis[mid].triOffset <= tri)
            lo = mid;
        else
            hi = mid - 1;
    }
    const MeshInstance &mi = mis[lo];
    const uint32_t prim = tri - mi.triOffset;

    float pos[3][3], nrm[3][3], tan[3][3], bit[3][3], uv[3][2];
#pragma unroll
    for (int k = 0; k < 3; k++)
    {
        // indices are relative to the geometry's first vertex (PT/Shaders/common.glsl:27-34)
        uint32_t index = indices[mi.indexOffset + prim * 3 + k];
        if (index >= mi.vertexLength)
        {
            // a malformed file: never read outside the geometry's vertices; the upload fails (PT_ERR_INVALID_ARGUMENT)
            atomicAdd(badIndexCount, 1u);
            index = 0;
        }
        const float *v = vertices + (size_t)(mi.vertexOffset + index) * 14;
        const float px = v[0], py = v[1], pz = v[2];
#pragma unroll
        for (int j = 0; j < 3; j++)
        {
            // same operation order as `vec4(p, 1) * transform`, unfused, so that the oracle and the
            // core intersect bit-identical triangles
            const float *P = mi.P + j * 4;
            pos[k][j] = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(px, P[0]), __fmul_rn(py, P[1])), __fmul_rn(pz, P[2])), P[3]);
            nrm[k][j] = mi.N[j * 3 + 0] * v[5] + mi.N[j * 3 + 1] * v[6] + mi.N[j * 3 + 2] * v[7];
            tan[k][j] = P[0] * v[8] + P[1] * v[9] + P[2] * v[10];
            bit[k][j] = P[0] * v[11] + P[1] * v[12] + P[2] * v[13];
        }
        uv[k][0] = v[3];
        uv[k][1] = v[4];
    }
    triPos[3 * (size_t)tri + 0] = make_float4(pos[0][0], pos[0][1], pos[0][2], __uint_as_float(tri));
    triPos[3 * (size_t)tri + 1] = make_float4(pos[1][0], pos[1][1], pos[1][2], __uint_as_float(mi.flags));
    triPos[3 * (size_t)tri + 2] = make_float4(pos[2][0], pos[2][1], pos[2][2], __uint_as_float(mi.materialId));

    TriShade ts;
    ts.a[0] = make_float4(nrm[0][0], nrm[0][1], nrm[0][2], nrm[1][0]);
    ts.a[1] = make_float4(nrm[1][1], nrm[1][2], nrm[2][0], nrm[2][1]);
    ts.a[2] = make_float4(nrm[2][2], tan[0][0], tan[0][1], tan[0][2]);
    ts.a[3] = make_float4(tan[1][0], tan[1][1], tan[1][2], tan[2][0]);
    ts.a[4] = make_float4(tan[2][1], tan[2][2], bit[0][0], bit[0][1]);
    ts.a[5] = make_float4(bit[0][2], bit[1][0], bit[1][1], bit[1][2]);
    ts.a[6] = make_float4(bit[2][0], bit[2][1], bit[2][2], uv[0][0]);
    ts.a[7] = make_float4(uv[0][1], uv[1][0], uv[1][1], uv[2][0]);
    ts.a[8] = make_float4(uv[2][1], __uint_as_float(mi.instance), __uint_as_float(mi.geometry), __uint_as_float(prim));
    const vec3 u0 = normalize(V3(nrm[0][0], nrm[0][1], nrm[0][2])), u1 = normalize(V3(nrm[1][0], nrm[1][1], nrm[1][2]));
    const vec3 u2 = normalize(V3(nrm[2][0], nrm[2][1], nrm[2][2]));
    const vec3 w0 = V3(pos[0][0], pos[0][1], pos[0][2]), w1 = V3(pos[1][0], pos[1][1], pos[1][2]);
    const vec3 w2 = V3(pos[2][0], pos[2][1], pos[2][2]);
    const vec3 g = normalize(cross(w1 - w0, w2 - w0));
    ts.a[9] = make_float4(u0.x, u0.y, u0.z, u1.x);
    ts.a[10] = make_float4(u1.y, u1.z, u2.x, u2.y);
    ts.a[11] = make_float4(u2.z, g.x, g.y, g.z);
    triShade[tri] = ts;

    Aabb b;
#pragma unroll
    for (int j = 0; j < 3; j++)
    {
        b.lo[j] = fminf(pos[0][j], fminf(pos[1][j], pos[2][j]));
        b.hi[j] = fmaxf(pos[0][j], fmaxf(pos[1][j], pos[2][j]));
    }
    boxes[tri] = b;
    // centroid bounds (of box centres), order-preserving uint encoding
#pragma unroll
    for (int j = 0; j < 3; j++)
    {
        const float c = 0.5f * (b.lo[j] + b.hi[j]);
        atomicMin(sceneBounds + j, floatFlip(c));
        atomicMax(sceneBounds + 3 + j, floatFlip(c));
    }
}

// ---------------------------------------------------------------------------------------------
// skinning.comp:21-50 — Renderer::RecordSkinningCommands (PT/Renderer/Renderer.cpp:854-890).
// One thread per animated vertex: blends the bone-transformed position / tangent frame with up to
// MaxBonesPerVertex = 4 weights (the loop stops once the weights reach 1).  bones[b] = the 12 floats
// of the bone's mat3x4 (three vec4 columns = rows of the 3x4 matrix) followed by the 9 of its normal
// matrix (inverse transpose of the linear part, precomputed on the host like the instances').
// The reference writes into a separate "out animated vertex" buffer per frame in flight; here the
// skinned vertices live behind the static ones in the one vertex buffer k_bake reads.
// ---------------------------------------------------------------------------------------------
#define PT_BONE_STRIDE 21
__global__ void k_skin(const float *__restrict__ animated, uint32_t count, const float *__restrict__ bones, uint32_t boneCount,
                       float *__restrict__ out)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count)
        return;
    const float *a = animated + (size_t)i * 22;
    const vec3 P = V3(a[0], a[1], a[2]), N = V3(a[5], a[6], a[7]), T = V3(a[8], a[9], a[10]), B = V3(a[11], a[12], a[13]);
    vec3 pos = V3(0.0f), nrm = V3(0.0f), tan = V3(0.0f), bit = V3(0.0f);
    float totalWeight = 0.0f;
    for (int k = 0; k < 4 && totalWeight < 1.0f; k++)
    {
        const uint32_t bone = min(__float_as_uint(a[14 + k]), boneCount - 1); // (an index past the UBO is undefined in GLSL)
        const float w = a[18 + k];
        const float *m = bones + (size_t)bone * PT_BONE_STRIDE;
        // vec4(v, 1 | 0) * mat3x4: component j = dot(v4, column j)
        // `boneWeight * vec4(Position, 1) * transform` groups from the left (skinning.comp:41): the WEIGHTED point
        // (w P, w) goes through the matrix
        auto xformWeightedPoint = [&](vec3 v, float vw) {
            return V3(((v.x * m[0] + v.y * m[1]) + v.z * m[2]) + vw * m[3], ((v.x * m[4] + v.y * m[5]) + v.z * m[6]) + vw * m[7],
                      ((v.x * m[8] + v.y * m[9]) + v.z * m[10]) + vw * m[11]);
        };
        auto xformDir = [&](vec3 v) {
            return V3(((v.x * m[0] + v.y * m[1]) + v.z * m[2]) + 0.0f * m[3], ((v.x * m[4] + v.y * m[5]) + v.z * m[6]) + 0.0f * m[7],
                      ((v.x * m[8] + v.y * m[9]) + v.z * m[10]) + 0.0f * m[11]);
        };
        const float *nm = m + 12;
        const vec3 nn = V3((N.x * nm[0] + N.y * nm[1]) + N.z * nm[2], (N.x * nm[3] + N.y * nm[4]) + N.z * nm[5],
                           (N.x * nm[6] + N.y * nm[7]) + N.z * nm[8]);
        pos = pos + xformWeightedPoint(w * P, w);
        tan = tan + w * normalize(xformDir(T));
        bit = bit + w * normalize(xformDir(B));
        nrm = nrm + w * normalize(nn);
        totalWeight += w;
    }
    float *o = out + (size_t)i * 14;
    o[0] = pos.x, o[1] = pos.y, o[2] = pos.z;
    o[3] = a[3], o[4] = a[4];
    o[5] = nrm.x, o[6] = nrm.y, o[7] = nrm.z;
    o[8] = tan.x, o[9] = tan.y, o[10] = tan.z;
    o[11] = bit.x, o[12] = bit.y, o[13] = bit.z;
}

__device__ __forceinline__ uint64_t expandBits21(uint64_t v)
{
    v &= 0x1fffffull;
    v = (v | v << 32) & 0x1f00000000ffffull;
    v = (v | v << 16) & 0x1f0000ff0000ffull;
    v = (v | v << 8) & 0x100f00f00f00f00full;
    v = (v | v << 4) & 0x10c30c30c30c30c3ull;
    v = (v | v << 2) & 0x1249249249249249ull;
    return v;
}

__global__ void k_morton(const Aabb *__restrict__ boxes, uint32_t n, const uint32_t *__restrict__ sceneBounds,
                         uint64_t *__restrict__ keys, uint32_t *__restrict__ values)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n)
        return;
    uint64_t code = 0;
#pragma unroll
    for (int j = 0; j < 3; j++)
    {
        const float lo = floatUnflip(sceneBounds[j]), hi = floatUnflip(sceneBounds[3 + j]);
        const float c = 0.5f * (boxes[i].lo[j] + boxes[i].hi[j]);
        const float ext = hi - lo;
        float f = ext > 0.0f ? (c - lo) / ext : 0.0f;
        f = fminf(fmaxf(f * 2097152.0f, 0.0f), 2097151.0f);
        code |= expandBits21((uint64_t)f) << (2 - j);
    }
    keys[i] = code;
    values[i] = i;
}

// ---------------------------------------------------------------------------------------------
// Reference splitting (early split clipping, Ernst & Greiner 2007, in the midpoint-subdivision form).
// A triangle whose bounding box is large compared with the space a primitive has in this scene — a big
// triangle lying diagonally, e.g. the randomly oriented alpha-tested cards of foliage — makes every
// box around it mostly empty, and in a dense soup of such triangles every ray walks through hundreds of
// overlapping boxes.  Such a triangle enters the BVH as 4^L REFERENCES, one per piece of its L-fold
// midpoint subdivision, each with the (slightly padded) box of its piece; all of them carry the PARENT's
// three corners, so the ray / triangle arithmetic, hit distances, barycentrics and ids are exactly what
// they are without splitting (a parent reached through two references is the same candidate twice: the
// closest-hit rule "t < best, or the same t and a smaller id" drops the repeat).
// ---------------------------------------------------------------------------------------------
#define PT_SPLIT_MAX_LEVEL 3

__global__ void k_split_count(const Aabb *__restrict__ boxes, uint32_t n, const uint32_t *__restrict__ sceneBounds, float threshold,
                              uint32_t *__restrict__ refCount)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n)
        return;
    // the space one primitive has: the volume of the scene (centroid bounds, padded) over the primitive count
    float ext[3];
    for (int j = 0; j < 3; j++)
        ext[j] = fmaxf(floatUnflip(sceneBounds[3 + j]) - floatUnflip(sceneBounds[j]), 1e-20f);
    const float share = ext[0] * ext[1] * ext[2] / (float)n;
    const Aabb b = boxes[i];
    const float v = (b.hi[0] - b.lo[0]) * (b.hi[1] - b.lo[1]) * (b.hi[2] - b.lo[2]);
    // every level of subdivision divides the box volume of a piece by 8 (and the summed volume by 2)
    uint32_t level = 0;
    float r = v / share;
    while (level < PT_SPLIT_MAX_LEVEL && r > threshold && isfinite(r))
    {
        level++;
        r *= 0.125f;
    }
    refCount[i] = 1u << (2 * level);
}

__global__ void k_split_emit(const float4 *__restrict__ triPos, const Aabb *__restrict__ boxes, uint32_t n,
                             const uint32_t *__restrict__ refCount, const uint32_t *__restrict__ refOffset, Aabb *__restrict__ refBoxes,
                             uint32_t *__restrict__ refTri)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n)
        return;
    const uint32_t count = refCount[i], first = refOffset[i];
    if (count == 1)
    {
        refBoxes[first] = boxes[i];
        refTri[first] = i;
        return;
    }
    const float4 q0 = triPos[3 * (size_t)i], q1 = triPos[3 * (size_t)i + 1], q2 = triPos[3 * (size_t)i + 2];
    const Aabb parent = boxes[i];
    for (uint32_t k = 0; k < count; k++)
    {
        float a[3] = { q0.x, q0.y, q0.z }, b[3] = { q1.x, q1.y, q1.z }, c[3] = { q2.x, q2.y, q2.z };
        // base-4 digits of k, most significant first: 0, 1, 2 = the corner piece at a, b, c; 3 = the middle piece
        for (uint32_t div = count >> 2; div >= 1; div >>= 2)
        {
            const uint32_t digit = (k / div) & 3u;
            float ab[3], bc[3], ca[3];
            for (int j = 0; j < 3; j++)
            {
                ab[j] = 0.5f * (a[j] + b[j]);
                bc[j] = 0.5f * (b[j] + c[j]);
                ca[j] = 0.5f * (c[j] + a[j]);
            }
            for (int j = 0; j < 3; j++)
            {
                const float na = digit == 0 ? a[j] : digit == 1 ? ab[j] : digit == 2 ? ca[j] : ab[j];
                const float nb = digit == 0 ? ab[j] : digit == 1 ? b[j] : digit == 2 ? bc[j] : bc[j];
                const float nc = digit == 0 ? ca[j] : digit == 1 ? bc[j] : digit == 2 ? c[j] : ca[j];
                a[j] = na, b[j] = nb, c[j] = nc;
            }
            if (div == 1)
                break;
        }
        Aabb r;
        for (int j = 0; j < 3; j++)
        {
            const float lo = fminf(a[j], fminf(b[j], c[j])), hi = fmaxf(a[j], fmaxf(b[j], c[j]));
            // the computed midpoints are within an ulp of the true edges: pad, and never beyond the parent's box
            const float pad = 4.0f * 1.1920929e-7f * fmaxf(fabsf(lo), fabsf(hi)) + 1e-30f;
            r.lo[j] = fmaxf(lo - pad, parent.lo[j]);
            r.hi[j] = fminf(hi + pad, parent.hi[j]);
        }
        refBoxes[first + k] = r;
        refTri[first + k] = i;
    }
}

// ---------------------------------------------------------------------------------------------
// LBVH (Karras 2012).  Nodes 0..n-2 internal, n-1..2n-2 leaves (leaf k <-> sorted primitive k).
// ---------------------------------------------------------------------------------------------
struct Bvh2
{
    int *left, *right, *parent;
    uint32_t *first, *last; // covered range of sorted primitives (LBVH only)
    uint32_t *count;        // primitives below the node
    Aabb *box;
    uint32_t *visit;
};

__device__ __forceinline__ int delta(const uint64_t *keys, int n, int i, int j)
{
    if (j < 0 || j >= n)
        return -1;
    const uint64_t a = keys[i], b = keys[j];
    if (a == b)
        return 64 + __clz(i ^ j);
    return __clzll(a ^ b);
}

__global__ void k_hierarchy(const uint64_t *__restrict__ keys, int n, Bvh2 t)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n - 1)
        return;
    const int d = (delta(keys, n, i, i + 1) - delta(keys, n, i, i - 1)) >= 0 ? 1 : -1;
    const int deltaMin = delta(keys, n, i, i - d);
    int lmax = 2;
    while (delta(keys, n, i, i + lmax * d) > deltaMin)
        lmax *= 2;
    int l = 0;
    for (int s = lmax / 2; s >= 1; s /= 2)
        if (delta(keys, n, i, i + (l + s) * d) > deltaMin)
            l += s;
    const int j = i + l * d;
    const int deltaNode = delta(keys, n, i, j);
    int s = 0;
    int tt = l;
    do
    {
        tt = (tt + 1) >> 1;
        if (delta(keys, n, i, i + (s + tt) * d) > deltaNode)
            s += tt;
    } while (tt > 1);
    const int gamma = i + s * d + min(d, 0);
    const int lo = min(i, j), hi = max(i, j);
    const int leftIdx = (lo == gamma) ? (n - 1 + gamma) : gamma;
    const int rightIdx = (hi == gamma + 1) ? (n - 1 + gamma + 1) : (gamma + 1);
    t.left[i] = leftIdx;
    t.right[i] = rightIdx;
    t.parent[leftIdx] = i;
    t.parent[rightIdx] = i;
    t.first[i] = lo;
    t.last[i] = hi;
    t.count[i] = (uint32_t)(hi - lo + 1);
    if (i == 0)
        t.parent[0] = -1;
}

__global__ void k_refit(const Aabb *__restrict__ primBoxes, const uint32_t *__restrict__ sortedIdx, int n, Bvh2 t)
{
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n)
        return;
    const int leaf = n - 1 + k;
    t.box[leaf] = primBoxes[sortedIdx[k]];
    t.first[leaf] = k;
    t.last[leaf] = k;
    t.count[leaf] = 1;
    int node = t.parent[leaf];
    while (node >= 0)
    {
        __threadfence();
        if (atomicAdd(t.visit + node, 1u) == 0)
            return; // the sibling will finish this node
        const Aabb a = t.box[t.left[node]], b = t.box[t.right[node]];
        Aabb m;
#pragma unroll
        for (int j = 0; j < 3; j++)
        {
            m.lo[j] = fminf(a.lo[j], b.lo[j]);
            m.hi[j] = fmaxf(a.hi[j], b.hi[j]);
        }
        t.box[node] = m;
        node = t.parent[node];
    }
}

__device__ __forceinline__ float halfArea(const Aabb &b)
{
    const float dx = b.hi[0] - b.lo[0], dy = b.hi[1] - b.lo[1], dz = b.hi[2] - b.lo[2];
    return dx * dy + dy * dz + dz * dx;
}

// ---------------------------------------------------------------------------------------------
// PLOC — parallel locally-ordered clustering (Meister & Bittner, TVCG 2018).  The clusters (at first
// the triangles, in Morton order) are merged bottom-up: every cluster looks for its nearest
// neighbour among the PT_PLOC radius clusters on either side of it in the array, "nearest" meaning
// the smallest surface area of the merged box; pairs that chose each other are merged into a new
// BVH2 node, the array is compacted, repeat until one cluster is left.  The result is close to a
// full-sweep SAH build in ray-tracing cost at a few ms per million triangles.
//
// Pairs are compared by the key (area, index distance, parity of the left index, left index): a
// total order both ends of a pair evaluate identically, so the globally smallest pair is always
// mutual (progress), and runs of identical boxes pair up as (0,1)(2,3)... instead of merging one
// pair per pass.
// ---------------------------------------------------------------------------------------------
#define PT_PLOC_BLOCK 256
#define PT_PLOC_MAX_RADIUS 64

__global__ void k_ploc_leaves(const Aabb *__restrict__ primBoxes, const uint32_t *__restrict__ sortedIdx, uint32_t n, Bvh2 t,
                              int *__restrict__ clusters)
{
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n)
        return;
    const uint32_t leaf = n - 1 + k;
    t.box[leaf] = primBoxes[sortedIdx[k]];
    t.count[leaf] = 1;
    clusters[k] = (int)leaf;
}

__global__ void __launch_bounds__(PT_PLOC_BLOCK)
    k_ploc_nearest(const int *__restrict__ clusters, uint32_t m, const Aabb *__restrict__ boxes, int radius,
                   uint32_t *__restrict__ nearest)
{
    __shared__ float sb[6][PT_PLOC_BLOCK + 2 * PT_PLOC_MAX_RADIUS];
    const int base = (int)(blockIdx.x * PT_PLOC_BLOCK) - radius;
    for (int k = threadIdx.x; k < PT_PLOC_BLOCK + 2 * radius; k += PT_PLOC_BLOCK)
    {
        const int j = base + k;
        if (j >= 0 && j < (int)m)
        {
            const Aabb b = boxes[clusters[j]];
            sb[0][k] = b.lo[0], sb[1][k] = b.lo[1], sb[2][k] = b.lo[2];
            sb[3][k] = b.hi[0], sb[4][k] = b.hi[1], sb[5][k] = b.hi[2];
        }
    }
    __syncthreads();
    const int i = (int)(blockIdx.x * PT_PLOC_BLOCK + threadIdx.x);
    if (i >= (int)m)
        return;
    const int li = (int)threadIdx.x + radius;
    const float lx = sb[0][li], ly = sb[1][li], lz = sb[2][li], hx = sb[3][li], hy = sb[4][li], hz = sb[5][li];
    float bestArea = INFINITY;
    int bestDist = 0x7fffffff, bestLeft = 0x7fffffff, bestJ = -1;
    const int j0 = max(0, i - radius), j1 = min((int)m - 1, i + radius);
    for (int j = j0; j <= j1; j++)
    {
        if (j == i)
            continue;
        const int lj = j - base;
        const float dx = fmaxf(hx, sb[3][lj]) - fminf(lx, sb[0][lj]);
        const float dy = fmaxf(hy, sb[4][lj]) - fminf(ly, sb[1][lj]);
        const float dz = fmaxf(hz, sb[5][lj]) - fminf(lz, sb[2][lj]);
        float area = dx * dy + dy * dz + dz * dx;
        if (!(area < INFINITY))
            area = INFINITY; // NaN / overflow: still a valid, symmetric key
        const int dist = abs(i - j), left = min(i, j);
        bool better = area < bestArea;
        if (area == bestArea)
        {
            if (dist != bestDist)
                better = dist < bestDist;
            else if ((left & 1) != (bestLeft & 1))
                better = (left & 1) == 0;
            else
                better = left < bestLeft;
        }
        if (better)
        {
            bestArea = area;
            bestDist = dist;
            bestLeft = left;
            bestJ = j;
        }
    }
    nearest[i] = (uint32_t)bestJ;
}

// flags[i] = (cluster i stays in the array) | (cluster i is the left end of a merging pair) << 32
__global__ void k_ploc_flags(const uint32_t *__restrict__ nearest, uint32_t m, unsigned long long *__restrict__ flags)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m)
        return;
    const uint32_t j = nearest[i];
    const bool mutual = nearest[j] == i;
    const unsigned long long keep = !(mutual && i > j), merger = mutual && i < j;
    flags[i] = keep | (merger << 32);
}

// scan[i] = exclusive prefix sum of flags: low word = position after compaction, high word = rank
// among this pass's merges.  Merge number q (counted over all passes) creates node n - 2 - q, so that
// the last merge creates the root, node 0.
__global__ void k_ploc_merge(const int *__restrict__ clusters, uint32_t m, const uint32_t *__restrict__ nearest,
                             const unsigned long long *__restrict__ flags, const unsigned long long *__restrict__ scan,
                             uint32_t n, uint32_t mergesBefore, Bvh2 t, int *__restrict__ clustersOut,
                             uint32_t *__restrict__ totals)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m)
        return;
    const unsigned long long f = flags[i], sc = scan[i];
    const uint32_t keep = (uint32_t)f & 1u, merger = (uint32_t)(f >> 32);
    const uint32_t pos = (uint32_t)sc, rank = (uint32_t)(sc >> 32);
    if (i == m - 1)
    {
        totals[0] = pos + keep;    // clusters left
        totals[1] = rank + merger; // merges of this pass
    }
    if (!keep)
        return;
    int node = clusters[i];
    if (merger)
    {
        const int other = clusters[nearest[i]];
        const int id = (int)(n - 2u - (mergesBefore + rank));
        const Aabb a = t.box[node], b = t.box[other];
        Aabb u;
#pragma unroll
        for (int j = 0; j < 3; j++)
        {
            u.lo[j] = fminf(a.lo[j], b.lo[j]);
            u.hi[j] = fmaxf(a.hi[j], b.hi[j]);
        }
        t.box[id] = u;
        t.left[id] = node;
        t.right[id] = other;
        t.count[id] = t.count[node] + t.count[other];
        node = id;
    }
    clustersOut[pos] = node;
}

// Writes one wide node from the exact child boxes (empty slots: lo = +inf, hi = -inf, ref = PT_CHILD_EMPTY).
__device__ __forceinline__ void writeWideNode(BvhNode *dst, const float lo[3][4], const float hi[3][4], const int ref[4])
{
    BvhNode out;
    float o[3], step[3];
    uint32_t qlo[3] = { 0, 0, 0 }, qhi[3] = { 0, 0, 0 };
    for (int j = 0; j < 3; j++)
    {
        float mn = INFINITY, mx = -INFINITY;
        for (int i = 0; i < 4; i++)
            if (ref[i] != PT_CHILD_EMPTY)
            {
                mn = fminf(mn, lo[j][i]);
                mx = fmaxf(mx, hi[j][i]);
            }
        if (!(mn <= mx) || !isfinite(mn) || !isfinite(mx)) // no children, or non-finite geometry: a box nothing hits
            mn = mx = 0.0f;
        // grid: 254 steps must span the node (one step of head room for the outward rounding below)
        int ex = 0;
        const float ext = mx - mn;
        (void)frexpf(fmaxf(ext / 254.0f, 1e-30f), &ex); // ext / 254 = m * 2^ex, m in [0.5, 1)  =>  2^ex >= ext / 254
        o[j] = mn;
        step[j] = ldexpf(1.0f, ex);
        for (int i = 0; i < 4; i++)
        {
            uint32_t a = 255u, b = 0u; // empty: entry plane beyond exit plane
            if (ref[i] != PT_CHILD_EMPTY && isfinite(lo[j][i]) && isfinite(hi[j][i]))
            {
                // outward rounding, verified with directed rounding: origin + a * step <= lo, origin + b * step >= hi
                int qa = (int)floorf((lo[j][i] - mn) / step[j]), qb = (int)ceilf((hi[j][i] - mn) / step[j]);
                qa = max(0, min(255, qa));
                qb = max(0, min(255, qb));
                while (qa > 0 && __fmaf_ru((float)qa, step[j], mn) > lo[j][i])
                    qa--;
                while (qb < 255 && __fmaf_rd((float)qb, step[j], mn) < hi[j][i])
                    qb++;
                a = (uint32_t)qa, b = (uint32_t)qb;
            }
            qlo[j] |= a << (8 * i);
            qhi[j] |= b << (8 * i);
        }
    }
    out.ox = o[0], out.oy = o[1], out.oz = o[2];
    out.sx = step[0], out.sy = step[1], out.sz = step[2];
    out.qlox = qlo[0], out.qloy = qlo[1], out.qloz = qlo[2];
    out.qhix = qhi[0], out.qhiy = qhi[1], out.qhiz = qhi[2];
    out.child = make_int4(ref[0], ref[1], ref[2], ref[3]);
    *dst = out;
}

// One work item = (BVH2 internal node, wide node index, first triangle of the node's range in the
// final order).  Children are opened largest-area first until the node is 4 wide; sub-trees of
// <= PT_MAX_LEAF_TRIS primitives become leaves.  The triangles are laid out depth first: child k
// starts where child k - 1 ends, and a leaf writes the source indices of its triangles to
// order[first ...] (k_gather moves the triangle positions afterwards).
__global__ void k_collapse(Bvh2 t, int n, const uint4 *__restrict__ work, uint32_t workCount, uint4 *__restrict__ next,
                           uint32_t *__restrict__ nextCount, BvhNode *__restrict__ nodes, uint32_t *__restrict__ nodeCount,
                           const uint32_t *__restrict__ sortedIdx, uint32_t *__restrict__ order)
{
    const uint32_t w = blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= workCount)
        return;
    const int src = (int)work[w].x;
    const uint32_t dst = work[w].y;
    uint32_t first = work[w].z;
    int c[4];
    int cc = 2;
    c[0] = t.left[src];
    c[1] = t.right[src];
    auto isLeaf = [&](int node) { return t.count[node] <= PT_MAX_LEAF_TRIS; };
    while (cc < 4)
    {
        int bestSlot = -1;
        float bestArea = -1.0f;
        for (int i = 0; i < cc; i++)
            if (!isLeaf(c[i]))
            {
                const float a = halfArea(t.box[c[i]]);
                if (a > bestArea)
                {
                    bestArea = a;
                    bestSlot = i;
                }
            }
        if (bestSlot < 0)
            break;
        const int open = c[bestSlot];
        c[bestSlot] = t.left[open];
        c[cc++] = t.right[open];
    }
    float lo[3][4], hi[3][4];
    int ref[4];
    for (int i = 0; i < 4; i++)
    {
        if (i >= cc)
        {
            for (int j = 0; j < 3; j++)
            {
                lo[j][i] = INFINITY;
                hi[j][i] = -INFINITY;
            }
            ref[i] = PT_CHILD_EMPTY;
            continue;
        }
        const Aabb b = t.box[c[i]];
        for (int j = 0; j < 3; j++)
        {
            lo[j][i] = b.lo[j];
            hi[j][i] = b.hi[j];
        }
        const uint32_t count = t.count[c[i]];
        if (isLeaf(c[i]))
        {
            ref[i] = encodeLeaf(first, count);
            // the (at most PT_MAX_LEAF_TRIS) triangles below c[i], left to right
            int stack[PT_MAX_LEAF_TRIS];
            int sp = 0, node = c[i];
            uint32_t out = first;
            for (;;)
            {
                if (node >= n - 1)
                {
                    order[out++] = sortedIdx[node - (n - 1)];
                    if (sp == 0)
                        break;
                    node = stack[--sp];
                }
                else
                {
                    stack[sp++] = t.right[node];
                    node = t.left[node];
                }
            }
        }
        else
        {
            const uint32_t idx = atomicAdd(nodeCount, 1u);
            ref[i] = (int)idx;
            next[atomicAdd(nextCount, 1u)] = make_uint4((uint32_t)c[i], idx, first, 0u);
        }
        first += count;
    }
    writeWideNode(nodes + dst, lo, hi, ref);
}

// root of a scene whose whole BVH2 is one leaf (1..PT_MAX_LEAF_TRIS primitives)
__global__ void k_single_leaf_root(const Aabb *__restrict__ primBoxes, const uint32_t *__restrict__ sortedIdx, uint32_t n,
                                   BvhNode *__restrict__ nodes)
{
    Aabb m;
    for (int j = 0; j < 3; j++)
    {
        m.lo[j] = INFINITY;
        m.hi[j] = -INFINITY;
    }
    for (uint32_t k = 0; k < n; k++)
        for (int j = 0; j < 3; j++)
        {
            m.lo[j] = fminf(m.lo[j], primBoxes[sortedIdx[k]].lo[j]);
            m.hi[j] = fmaxf(m.hi[j], primBoxes[sortedIdx[k]].hi[j]);
        }
    float lo[3][4], hi[3][4];
    int ref[4] = { encodeLeaf(0, n), PT_CHILD_EMPTY, PT_CHILD_EMPTY, PT_CHILD_EMPTY };
    for (int j = 0; j < 3; j++)
        for (int i = 0; i < 4; i++)
        {
            lo[j][i] = i == 0 ? m.lo[j] : INFINITY;
            hi[j][i] = i == 0 ? m.hi[j] : -INFINITY;
        }
    writeWideNode(nodes, lo, hi, ref);
}

__global__ void k_gather(const uint32_t *__restrict__ sortedIdx, const uint32_t *__restrict__ refTri, uint32_t n,
                         const float4 *__restrict__ posIn, float4 *__restrict__ posOut)
{
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n)
        return;
    // leaf-order position k holds reference sortedIdx[k], i.e. (a copy of) its parent triangle
    const uint32_t src = refTri ? refTri[sortedIdx[k]] : sortedIdx[k];
    posOut[3 * (size_t)k + 0] = posIn[3 * (size_t)src + 0];
    posOut[3 * (size_t)k + 1] = posIn[3 * (size_t)src + 1];
    posOut[3 * (size_t)k + 2] = posIn[3 * (size_t)src + 2];
}


// Stream-ordered allocation from the device's default memory pool (release threshold raised at
// pt_context_create): the temporaries and outputs of buildAccel.  A second build — pt_scene_update,
// once per animated frame — gets its ~20 buffers back from the pool without a driver call; with
// cudaMalloc / cudaFree a 2 M-triangle rebuild took 90-600 ms of which 6 ms were kernels.
template <typename T> pt_status devAllocPool(Context *ctx, T **ptr, size_t count, std::vector<void *> &owner)
{
    *ptr = nullptr;
    if (count == 0)
        count = 1;
    PT_CUDA_CHECK(ctx, poolAlloc(ctx, (void **)ptr, count * sizeof(T), ctx->stream));
    owner.push_back(*ptr);
    return PT_OK;
}

template <typename T> pt_status devAlloc(Context *ctx, T **ptr, size_t count, std::vector<void *> &owner)
{
    *ptr = nullptr;
    if (count == 0)
        count = 1;
    PT_CUDA_CHECK(ctx, cudaMalloc((void **)ptr, count * sizeof(T)));
    owner.push_back(*ptr);
    return PT_OK;
}

// The normal matrix of sampling.glsl:12 / skinning.comp:44, `transpose(inverse(mat4(transform)))`, for
// a 3x4 row-major affine matrix P — evaluated in fp32 with the very operation order of the glm the
// reference vendors (glm/detail/func_matrix.inl, compute_inverse<4, 4>: 2x2 sub-determinants, cofactor
// columns a*b - c*d + e*f, pairwise determinant sum, one multiply by 1 / det), which is also what the
// oracle and the compiled-GLSL reference (oracle/_ref/libglsl_ref.so) do.  (A double-precision 3x3
// inverse is more accurate but rounds differently in the last bit; on scenes modelled in millimetres
// that last bit decides whether a shadow ray leaves its own triangle, i.e. whole pixels.)
// mat4(transform) has the ROWS of P as its columns.  N[j*3 + i] = inverse(m)[i][j]:
// world normal_j = sum_i N[j*3 + i] * n_i  (= (vec4(n, 0) * transpose(inverse(m))).xyz).
void normalMatrix(const float P[12], float N[9])
{
    const float m[4][4] = { { P[0], P[1], P[2], P[3] }, { P[4], P[5], P[6], P[7] }, { P[8], P[9], P[10], P[11] }, { 0.0f, 0.0f, 0.0f, 1.0f } };
    // volatile: one rounding per operation whatever the host compiler would like to contract
    auto dop = [](float a, float b, float c, float d) {
        const volatile float ab = a * b, cd = c * d;
        const volatile float r = ab - cd;
        return (float)r;
    };
    const float Coef00 = dop(m[2][2], m[3][3], m[3][2], m[2][3]), Coef02 = dop(m[1][2], m[3][3], m[3][2], m[1][3]);
    const float Coef03 = dop(m[1][2], m[2][3], m[2][2], m[1][3]), Coef04 = dop(m[2][1], m[3][3], m[3][1], m[2][3]);
    const float Coef06 = dop(m[1][1], m[3][3], m[3][1], m[1][3]), Coef07 = dop(m[1][1], m[2][3], m[2][1], m[1][3]);
    const float Coef08 = dop(m[2][1], m[3][2], m[3][1], m[2][2]), Coef10 = dop(m[1][1], m[3][2], m[3][1], m[1][2]);
    const float Coef11 = dop(m[1][1], m[2][2], m[2][1], m[1][2]), Coef12 = dop(m[2][0], m[3][3], m[3][0], m[2][3]);
    const float Coef14 = dop(m[1][0], m[3][3], m[3][0], m[1][3]), Coef15 = dop(m[1][0], m[2][3], m[2][0], m[1][3]);
    const float Coef16 = dop(m[2][0], m[3][2], m[3][0], m[2][2]), Coef18 = dop(m[1][0], m[3][2], m[3][0], m[1][2]);
    const float Coef19 = dop(m[1][0], m[2][2], m[2][0], m[1][2]), Coef20 = dop(m[2][0], m[3][1], m[3][0], m[2][1]);
    const float Coef22 = dop(m[1][0], m[3][1], m[3][0], m[1][1]), Coef23 = dop(m[1][0], m[2][1], m[2][0], m[1][1]);
    const float Fac0[4] = { Coef00, Coef00, Coef02, Coef03 }, Fac1[4] = { Coef04, Coef04, Coef06, Coef07 };
    const float Fac2[4] = { Coef08, Coef08, Coef10, Coef11 }, Fac3[4] = { Coef12, Coef12, Coef14, Coef15 };
    const float Fac4[4] = { Coef16, Coef16, Coef18, Coef19 }, Fac5[4] = { Coef20, Coef20, Coef22, Coef23 };
    const float Vec0[4] = { m[1][0], m[0][0], m[0][0], m[0][0] }, Vec1[4] = { m[1][1], m[0][1], m[0][1], m[0][1] };
    const float Vec2[4] = { m[1][2], m[0][2], m[0][2], m[0][2] }, Vec3[4] = { m[1][3], m[0][3], m[0][3], m[0][3] };
    // a*b - c*d + e*f
    auto col = [](const float *a, const float *b, const float *c, const float *d, const float *e, const float *f, const float *sign,
                  float *out) {
        for (int k = 0; k < 4; k++)
        {
            const volatile float ab = a[k] * b[k], cd = c[k] * d[k], ef = e[k] * f[k];
            const volatile float t = ab - cd;
            const volatile float r = t + ef;
            out[k] = r * sign[k];
        }
    };
    const float SignA[4] = { +1.0f, -1.0f, +1.0f, -1.0f }, SignB[4] = { -1.0f, +1.0f, -1.0f, +1.0f };
    float Inv[4][4];
    col(Vec1, Fac0, Vec2, Fac1, Vec3, Fac2, SignA, Inv[0]);
    col(Vec0, Fac0, Vec2, Fac3, Vec3, Fac4, SignB, Inv[1]);
    col(Vec0, Fac1, Vec1, Fac3, Vec3, Fac5, SignA, Inv[2]);
    col(Vec0, Fac2, Vec1, Fac4, Vec2, Fac5, SignB, Inv[3]);
    const volatile float d0 = m[0][0] * Inv[0][0], d1 = m[0][1] * Inv[1][0], d2 = m[0][2] * Inv[2][0], d3 = m[0][3] * Inv[3][0];
    const volatile float s01 = d0 + d1, s23 = d2 + d3;
    const volatile float det = s01 + s23;
    const float inv = 1.0f / det;
    for (int j = 0; j < 3; j++)
        for (int i = 0; i < 3; i++)
            N[j * 3 + i] = Inv[i][j] * inv;
}


void freeAccel(Context *ctx)
{
    for (void *p : ctx->accelAllocs)
        cudaFreeAsync(p, ctx->stream);
    ctx->accelAllocs.clear();
    ctx->scene.nodes = nullptr;
    ctx->scene.triPos = nullptr;
    ctx->scene.triShade = nullptr;
}

// Bakes the flattened mesh instances into world-space triangles and builds the BVH over them, all
// on the GPU, from the device-resident vertex / index buffers.  Replaces the previous triangle
// streams and nodes of the scene (pt_scene_upload calls it once, pt_scene_update per changed frame).
pt_status buildAccel(Context *ctx, const std::vector<MeshInstance> &mis, uint32_t n)
{
    freeAccel(ctx);
    DeviceScene &s = ctx->scene;
    std::vector<void *> temp;
    auto freeTemp = [&]() {
        for (void *p : temp)
            cudaFreeAsync(p, ctx->stream);
        temp.clear();
    };
#define PT_TRY(expr)                                                                                                  \
    do                                                                                                                \
    {                                                                                                                 \
        const pt_status st__ = (expr);                                                                                \
        if (st__ != PT_OK)                                                                                            \
        {                                                                                                             \
            freeTemp();                                                                                               \
            return st__;                                                                                              \
        }                                                                                                             \
    } while (0)
    s.triCount = n;
    ctx->nodeCount = 0;
    ctx->bvhBytes = 0;
    if (n > 0)
    {
        // ---- bake -------------------------------------------------------------------------
        const float *dVertices = ctx->dVertices;
        const uint32_t *dIndices = ctx->dIndices;
        MeshInstance *dMis;
        float4 *posUnsorted;
        TriShade *triShade;
        Aabb *primBoxes;
        uint32_t *sceneBounds;
        PT_TRY(devAllocPool(ctx, &dMis, mis.size(), temp));
        PT_TRY(devAllocPool(ctx, &posUnsorted, (size_t)n * 3, temp));
        PT_TRY(devAllocPool(ctx, &triShade, (size_t)n, ctx->accelAllocs)); // stays: the scene's shading records
        PT_TRY(devAllocPool(ctx, &primBoxes, (size_t)n, temp));
        PT_TRY(devAllocPool(ctx, &sceneBounds, 7, temp)); // 6 bounds + the bad-index counter of k_bake
        PT_CUDA_CHECK(ctx, cudaMemcpyAsync(dMis, mis.data(), mis.size() * sizeof(MeshInstance), cudaMemcpyHostToDevice, ctx->stream));
        const uint32_t boundsInit[7] = { 0xffffffffu, 0xffffffffu, 0xffffffffu, 0u, 0u, 0u, 0u };
        PT_CUDA_CHECK(ctx, cudaMemcpyAsync(sceneBounds, boundsInit, sizeof(boundsInit), cudaMemcpyHostToDevice, ctx->stream));
        PT_CUDA_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
        const uint32_t T = 256;
        uint32_t G = (n + T - 1) / T;
        k_bake<<<G, T, 0, ctx->stream>>>(dMis, (uint32_t)mis.size(), dVertices, dIndices, n, posUnsorted, triShade,
                                         primBoxes, sceneBounds, sceneBounds + 6);
        {
            uint32_t badIndices = 0;
            PT_CUDA_CHECK(ctx, cudaMemcpyAsync(&badIndices, sceneBounds + 6, 4, cudaMemcpyDeviceToHost, ctx->stream));
            PT_CUDA_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
            if (badIndices != 0)
            {
                freeTemp();
                return fail(ctx, PT_ERR_INVALID_ARGUMENT, "pt_scene_upload", "an index is not below its geometry's vertex_length");
            }
        }

        // ---- reference splitting (k_split_*): from here on `n` counts references ---------------------
        uint32_t *refTri = nullptr;
        ctx->triangleCount = n;
        if (ctx->splitThreshold > 0.0f && n > PT_MAX_LEAF_TRIS)
        {
            uint32_t *refCount, *refOffset;
            PT_TRY(devAllocPool(ctx, &refCount, (size_t)n + 1, temp));
            PT_TRY(devAllocPool(ctx, &refOffset, (size_t)n + 1, temp));
            PT_CUDA_CHECK(ctx, cudaMemsetAsync(refCount + n, 0, 4, ctx->stream));
            k_split_count<<<G, T, 0, ctx->stream>>>(primBoxes, n, sceneBounds, ctx->splitThreshold, refCount);
            size_t scanBytes = 0;
            cub::DeviceScan::ExclusiveSum(nullptr, scanBytes, refCount, refOffset, (int)n + 1, ctx->stream);
            uint8_t *scanTemp;
            PT_TRY(devAllocPool(ctx, &scanTemp, scanBytes, temp));
            PT_CUDA_CHECK(ctx, cub::DeviceScan::ExclusiveSum(scanTemp, scanBytes, refCount, refOffset, (int)n + 1, ctx->stream));
            uint32_t total = 0;
            PT_CUDA_CHECK(ctx, cudaMemcpyAsync(&total, refOffset + n, 4, cudaMemcpyDeviceToHost, ctx->stream));
            PT_CUDA_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
            if (total > n && (uint64_t)total < (1ull << 29))
            {
                Aabb *refBoxes;
                PT_TRY(devAllocPool(ctx, &refBoxes, (size_t)total, temp));
                PT_TRY(devAllocPool(ctx, &refTri, (size_t)total, temp));
                k_split_emit<<<G, T, 0, ctx->stream>>>(posUnsorted, primBoxes, n, refCount, refOffset, refBoxes, refTri);
                primBoxes = refBoxes;
                n = total;
                G = (n + T - 1) / T;
            }
        }
        s.triCount = n;

        // ---- Morton codes + sort ------------------------------------------------------------
        uint64_t *keysIn, *keysOut;
        uint32_t *valsIn, *valsOut;
        PT_TRY(devAllocPool(ctx, &keysIn, (size_t)n, temp));
        PT_TRY(devAllocPool(ctx, &keysOut, (size_t)n, temp));
        PT_TRY(devAllocPool(ctx, &valsIn, (size_t)n, temp));
        PT_TRY(devAllocPool(ctx, &valsOut, (size_t)n, temp));
        k_morton<<<G, T, 0, ctx->stream>>>(primBoxes, n, sceneBounds, keysIn, valsIn);
        size_t sortBytes = 0;
        cub::DeviceRadixSort::SortPairs(nullptr, sortBytes, keysIn, keysOut, valsIn, valsOut, (int)n, 0, 63, ctx->stream);
        uint8_t *sortTemp;
        PT_TRY(devAllocPool(ctx, &sortTemp, sortBytes, temp));
        PT_CUDA_CHECK(ctx, cub::DeviceRadixSort::SortPairs(sortTemp, sortBytes, keysIn, keysOut, valsIn, valsOut, (int)n, 0,
                                                           63, ctx->stream));

        // ---- hierarchy ------------------------------------------------------------------------
        BvhNode *wide;
        const uint32_t wideCapacity = std::max(1u, n); // <= n - 1 internal nodes (+ 1 for tiny scenes)
        PT_TRY(devAllocPool(ctx, &wide, (size_t)wideCapacity, temp));
        uint32_t wideCount = 1;
        uint32_t *order = valsOut; // source index of the triangle at every position of the final order
        if (n <= PT_MAX_LEAF_TRIS)
        {
            k_single_leaf_root<<<1, 1, 0, ctx->stream>>>(primBoxes, valsOut, n, wide);
            ctx->bvhMaxDepth = 1;
        }
        else
        {
            Bvh2 t;
            const size_t nodes2 = 2 * (size_t)n - 1;
            PT_TRY(devAllocPool(ctx, &t.left, (size_t)n, temp));
            PT_TRY(devAllocPool(ctx, &t.right, (size_t)n, temp));
            PT_TRY(devAllocPool(ctx, &t.count, nodes2, temp));
            PT_TRY(devAllocPool(ctx, &t.box, nodes2, temp));
            if (ctx->bvhBuilder == 0)
            {
                PT_TRY(devAllocPool(ctx, &t.parent, nodes2, temp));
                PT_TRY(devAllocPool(ctx, &t.first, nodes2, temp));
                PT_TRY(devAllocPool(ctx, &t.last, nodes2, temp));
                PT_TRY(devAllocPool(ctx, &t.visit, (size_t)n, temp));
                PT_CUDA_CHECK(ctx, cudaMemsetAsync(t.visit, 0, (size_t)n * 4, ctx->stream));
                k_hierarchy<<<G, T, 0, ctx->stream>>>(keysOut, (int)n, t);
                k_refit<<<G, T, 0, ctx->stream>>>(primBoxes, valsOut, (int)n, t);
            }
            else
            {
                t.parent = nullptr;
                t.first = t.last = t.visit = nullptr;
                const int radius = (int)std::min<uint32_t>(PT_PLOC_MAX_RADIUS, std::max<uint32_t>(1u, ctx->plocRadius));
                int *clusters[2];
                uint32_t *nearest, *totals;
                unsigned long long *flags, *scan;
                PT_TRY(devAllocPool(ctx, &clusters[0], (size_t)n, temp));
                PT_TRY(devAllocPool(ctx, &clusters[1], (size_t)n, temp));
                PT_TRY(devAllocPool(ctx, &nearest, (size_t)n, temp));
                PT_TRY(devAllocPool(ctx, &flags, (size_t)n, temp));
                PT_TRY(devAllocPool(ctx, &scan, (size_t)n, temp));
                PT_TRY(devAllocPool(ctx, &totals, 2, temp));
                size_t scanBytes = 0;
                cub::DeviceScan::ExclusiveSum(nullptr, scanBytes, flags, scan, (int)n, ctx->stream);
                uint8_t *scanTemp;
                PT_TRY(devAllocPool(ctx, &scanTemp, scanBytes, temp));
                k_ploc_leaves<<<G, T, 0, ctx->stream>>>(primBoxes, valsOut, n, t, clusters[0]);
                uint32_t m = n, merges = 0, passes = 0;
                int cur = 0;
                while (m > 1)
                {
                    const uint32_t gb = (m + PT_PLOC_BLOCK - 1) / PT_PLOC_BLOCK;
                    k_ploc_nearest<<<gb, PT_PLOC_BLOCK, 0, ctx->stream>>>(clusters[cur], m, t.box, radius, nearest);
                    k_ploc_flags<<<gb, PT_PLOC_BLOCK, 0, ctx->stream>>>(nearest, m, flags);
                    PT_CUDA_CHECK(ctx, cub::DeviceScan::ExclusiveSum(scanTemp, scanBytes, flags, scan, (int)m, ctx->stream));
                    k_ploc_merge<<<gb, PT_PLOC_BLOCK, 0, ctx->stream>>>(clusters[cur], m, nearest, flags, scan, n, merges, t,
                                                                        clusters[cur ^ 1], totals);
                    uint32_t h[2] = { 0, 0 };
                    PT_CUDA_CHECK(ctx, cudaMemcpyAsync(h, totals, 8, cudaMemcpyDeviceToHost, ctx->stream));
                    PT_CUDA_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
                    if (h[1] == 0 || h[0] + h[1] != m || ++passes > 100000)
                    {
                        freeTemp();
                        return fail(ctx, PT_ERR_CUDA, "pt_scene_upload", "PLOC made no progress (internal error)");
                    }
                    m = h[0];
                    merges += h[1];
                    cur ^= 1;
                }
                ctx->bvhBuildPasses = passes;
            }

            uint4 *work[2];
            uint32_t *counters; // [0] node count, [1], [2] work counts
            PT_TRY(devAllocPool(ctx, &work[0], (size_t)n, temp));
            PT_TRY(devAllocPool(ctx, &work[1], (size_t)n, temp));
            PT_TRY(devAllocPool(ctx, &counters, 3, temp));
            PT_TRY(devAllocPool(ctx, &order, (size_t)n, temp));
            const uint4 rootItem = make_uint4(0u, 0u, 0u, 0u);
            const uint32_t initCounters[3] = { 1u, 0u, 0u };
            PT_CUDA_CHECK(ctx, cudaMemcpyAsync(work[0], &rootItem, sizeof(rootItem), cudaMemcpyHostToDevice, ctx->stream));
            PT_CUDA_CHECK(ctx, cudaMemcpyAsync(counters, initCounters, sizeof(initCounters), cudaMemcpyHostToDevice, ctx->stream));
            PT_CUDA_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
            uint32_t workCount = 1;
            int cur = 0;
            ctx->bvhMaxDepth = 0;
            while (workCount > 0)
            {
                ctx->bvhMaxDepth++; // one pass of the collapse = one level of the wide tree
                PT_CUDA_CHECK(ctx, cudaMemsetAsync(counters + 1 + (cur ^ 1), 0, 4, ctx->stream));
                k_collapse<<<(workCount + 127) / 128, 128, 0, ctx->stream>>>(t, (int)n, work[cur], workCount, work[cur ^ 1],
                                                                             counters + 1 + (cur ^ 1), wide, counters, valsOut,
                                                                             order);
                PT_CUDA_CHECK(ctx, cudaMemcpyAsync(&workCount, counters + 1 + (cur ^ 1), 4, cudaMemcpyDeviceToHost, ctx->stream));
                PT_CUDA_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
                cur ^= 1;
            }
            PT_CUDA_CHECK(ctx, cudaMemcpyAsync(&wideCount, counters, 4, cudaMemcpyDeviceToHost, ctx->stream));
            PT_CUDA_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
        }

        // ---- final triangle streams, in leaf order ------------------------------------------------
        float4 *triPos;
        PT_TRY(devAllocPool(ctx, &triPos, (size_t)n * 3, ctx->accelAllocs));
        k_gather<<<G, T, 0, ctx->stream>>>(order, refTri, n, posUnsorted, triPos);
        s.triPos = triPos;
        s.triShade = triShade;
        BvhNode *nodes;
        PT_TRY(devAllocPool(ctx, &nodes, (size_t)wideCount, ctx->accelAllocs));
        PT_CUDA_CHECK(ctx, cudaMemcpyAsync(nodes, wide, (size_t)wideCount * sizeof(BvhNode), cudaMemcpyDeviceToDevice, ctx->stream));
        s.nodes = nodes;
        ctx->nodeCount = wideCount;
        ctx->bvhBytes = (uint64_t)wideCount * sizeof(BvhNode) + (uint64_t)n * 48 + ctx->triangleCount * sizeof(TriShade);
        ctx->referenceCount = n;
    }
    PT_CUDA_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    PT_CUDA_CHECK(ctx, cudaGetLastError());
    freeTemp();
    return PT_OK;
#undef PT_TRY
}

// Uploads the bone matrices (+ their normal matrices) and re-skins every animated vertex into its
// place behind the static vertices (Renderer::RecordSkinningCommands).
pt_status skinAnimatedVertices(Context *ctx, const float *boneTransforms)
{
    const SceneTopology &t = ctx->topo;
    std::vector<float> bones((size_t)t.boneCount * PT_BONE_STRIDE);
    for (uint32_t b = 0; b < t.boneCount; b++)
    {
        const float *m = boneTransforms + 12 * (size_t)b;
        float *o = bones.data() + (size_t)b * PT_BONE_STRIDE;
        std::memcpy(o, m, 48);
        normalMatrix(m, o + 12);
    }
    PT_CUDA_CHECK(ctx, cudaMemcpyAsync(ctx->dBones, bones.data(), bones.size() * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    const uint32_t n = (uint32_t)t.animatedVertexCount;
    k_skin<<<(n + 255) / 256, 256, 0, ctx->stream>>>(ctx->dAnimatedVertices, n, ctx->dBones, t.boneCount,
                                                     const_cast<float *>(ctx->dVertices) + (size_t)t.vertexCount * 14);
    PT_CUDA_CHECK(ctx, cudaGetLastError());
    PT_CUDA_CHECK(ctx, cudaStreamSynchronize(ctx->stream)); // `bones` is a local
    return PT_OK;
}

// P = Instance * Mesh with the evaluation order of `mat4(transforms[i]) * gl_ObjectToWorld3x4EXT`
// (PT/Shaders/sampling.glsl:7); A = the mesh transform, B = the instance transform, both as 3x4 rows
void composeTransform(const float *A, const float *B, float P[12])
{
    for (int j = 0; j < 3; j++)
        for (int c = 0; c < 4; c++)
        {
            float v = A[0 * 4 + c] * B[j * 4 + 0] + A[1 * 4 + c] * B[j * 4 + 1];
            v = v + A[2 * 4 + c] * B[j * 4 + 2];
            if (c == 3)
                v = v + 1.0f * B[j * 4 + 3];
            P[j * 4 + c] = v;
        }
}

// Flattens instances x meshes into one MeshInstance per (instance, mesh) pair with its baked
// object-to-world and normal matrices (host, tiny).
pt_status flattenInstances(Context *ctx, const SceneTopology &t, std::vector<MeshInstance> &mis, bool &hasAlpha)
{
    mis.clear();
    uint64_t triTotal = 0;
    hasAlpha = false;
    for (uint32_t ii = 0; ii < (uint32_t)t.instances.size(); ii++)
    {
        const pt_instance &inst = t.instances[ii];
        if (inst.model_index >= t.models.size())
            return fail(ctx, PT_ERR_INVALID_ARGUMENT, "pt_scene_upload", "instance.model_index out of range");
        const pt_model &model = t.models[inst.model_index];
        for (uint32_t mi = 0; mi < model.mesh_count; mi++)
        {
            if (model.mesh_offset + mi >= t.meshRecords.size())
                return fail(ctx, PT_ERR_INVALID_ARGUMENT, "pt_scene_upload", "model mesh range out of range");
            const pt_mesh_record &rec = t.meshRecords[model.mesh_offset + mi];
            if (rec.geometry_index >= t.geometries.size() || rec.transform_index >= t.transforms.size() / 12)
                return fail(ctx, PT_ERR_INVALID_ARGUMENT, "pt_scene_upload", "mesh record index out of range");
            const pt_geometry &g = t.geometries[rec.geometry_index];
            const bool animated = !t.geometryIsAnimated.empty() && t.geometryIsAnimated[rec.geometry_index] != 0;
            if ((uint64_t)g.index_offset + g.index_length > (animated ? t.animatedIndexCount : t.indexCount) ||
                (uint64_t)g.vertex_offset + g.vertex_length > (animated ? t.animatedVertexCount : t.vertexCount))
                return fail(ctx, PT_ERR_INVALID_ARGUMENT, "pt_scene_upload", "geometry range out of range");
            const uint32_t type = rec.material_id & 0xffu, index = rec.material_id >> 8;
            const uint32_t limit = type == 0 ? t.materialCount[0] : type == 1 ? t.materialCount[1]
                                                                  : type == 2   ? t.materialCount[2]
                                                                                : 0xffffffffu;
            if (index >= limit)
                return fail(ctx, PT_ERR_INVALID_ARGUMENT, "pt_scene_upload", "material index out of range");
            MeshInstance m = {};
            composeTransform(t.transforms.data() + 12 * (size_t)rec.transform_index, inst.transform, m.P);
            normalMatrix(m.P, m.N);
            m.triOffset = (uint32_t)triTotal;
            m.triCount = g.index_length / 3;
            // skinned vertices / animated indices sit behind the static ones in the device buffers
            m.vertexOffset = g.vertex_offset + (animated ? (uint32_t)t.vertexCount : 0u);
            m.indexOffset = g.index_offset + (animated ? (uint32_t)t.indexCount : 0u);
            m.vertexLength = g.vertex_length;
            m.instance = ii;
            m.geometry = mi;
            m.materialId = rec.material_id;
            m.flags = g.is_opaque ? PT_TRI_FLAG_OPAQUE : 0u;
            {
                // facing is decided in OBJECT space = the BLAS's space, after the mesh transform and before the
                // instance transform (gl_RayFlagsCullBackFacingTrianglesEXT, Debug/debugRaygen.rgen:32-35)
                const float *I = inst.transform;
                const double det = (double)I[0] * ((double)I[5] * I[10] - (double)I[6] * I[9]) -
                                   (double)I[1] * ((double)I[4] * I[10] - (double)I[6] * I[8]) +
                                   (double)I[2] * ((double)I[4] * I[9] - (double)I[5] * I[8]);
                if (det < 0.0)
                    m.flags |= PT_TRI_FLAG_MIRRORED;
            }
            hasAlpha |= !g.is_opaque;
            if (m.triCount == 0)
                continue;
            triTotal += m.triCount;
            mis.push_back(m);
        }
    }
    if (triTotal >= (1ull << 29))
        return fail(ctx, PT_ERR_UNSUPPORTED, "pt_scene_upload", "more than 2^29 instanced triangles");
    return PT_OK;

}

} // namespace

// PT_TEST_TRANSFORM_VERTEX: the host half of the vertex transform (flattenInstances' matrices)
void testComposeTransform(const float *meshRows, const float *instanceRows, float P[12], float N[9])
{
    composeTransform(meshRows, instanceRows, P);
    normalMatrix(P, N);
}

void freeScene(Context *ctx)
{
    freeEmitters(ctx);
    freeAccel(ctx);
    if (ctx->stream)
    {
        // hand the pool's cached blocks back to the driver: the next scene may be of another size
        cudaStreamSynchronize(ctx->stream);
        if (ctx->memPool)
            cudaMemPoolTrimTo(ctx->memPool, 0);
    }
    for (void *p : ctx->sceneAllocs)
        cudaFree(p);
    ctx->sceneAllocs.clear();
    ctx->hostTextures.clear();
    ctx->hasScene = false;
    ctx->scene = DeviceScene {};
}

pt_status uploadTextureSlot(Context *ctx, uint32_t slot, const pt_texture_desc *tex)
{
    if (!ctx->hasScene)
        return fail(ctx, PT_ERR_NO_SCENE, "pt_texture_upload", "no scene uploaded");
    if (!tex || slot >= ctx->hostTextures.size())
        return fail(ctx, PT_ERR_INVALID_ARGUMENT, "pt_texture_upload", "slot out of range");
    DevTexture t;
    void *mem = nullptr;
    const pt_status st = createTexture(ctx, *tex, t, &mem, slot >= PT_SCENE_TEXTURE_OFFSET);
    if (st != PT_OK)
        return st;
    // the old allocation stays owned by the scene until the next scene upload
    ctx->sceneAllocs.push_back(mem);
    ctx->hostTextures[slot] = t;
    ctx->emittersValid = false; // an emissive texture may have changed
    PT_CUDA_CHECK(ctx, cudaMemcpyAsync(const_cast<DevTexture *>(ctx->scene.textures) + slot, &t, sizeof(t),
                                       cudaMemcpyHostToDevice, ctx->stream));
    PT_CUDA_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    return PT_OK;
}

pt_status uploadScene(Context *ctx, const pt_scene_desc *d)
{
    if (!d)
        return fail(ctx, PT_ERR_INVALID_ARGUMENT, "pt_scene_upload", "scene is NULL");
    if (d->point_light_count > PT_MAX_LIGHT_COUNT)
        return fail(ctx, PT_ERR_INVALID_ARGUMENT, "pt_scene_upload", "more than 64 point lights");
    if (d->transform_count == 0 || !d->transforms)
        return fail(ctx, PT_ERR_INVALID_ARGUMENT, "pt_scene_upload", "transforms[0] (identity) is required");
    if ((d->vertex_count && !d->vertices) || (d->index_count && !d->indices) || (d->geometry_count && !d->geometries) ||
        (d->mesh_record_count && !d->mesh_records) || (d->model_count && !d->models) ||
        (d->instance_count && !d->instances) || (d->texture_count && !d->textures) ||
        (d->mr_material_count && !d->mr_materials) || (d->sg_material_count && !d->sg_materials) ||
        (d->phong_material_count && !d->phong_materials) || (d->point_light_count && !d->point_lights))
        return fail(ctx, PT_ERR_INVALID_ARGUMENT, "pt_scene_upload", "array pointer is NULL with a non-zero count");

    if (d->geometry_is_animated &&
        ((d->animated_vertex_count && !d->animated_vertices) || (d->animated_index_count && !d->animated_indices) ||
         d->bone_count == 0 || !d->bone_transforms))
        return fail(ctx, PT_ERR_INVALID_ARGUMENT, "pt_scene_upload", "animated geometries need animated vertices, indices and bone transforms");
    if (d->vertex_count + (d->geometry_is_animated ? d->animated_vertex_count : 0) >= (1ull << 32) ||
        d->index_count + (d->geometry_is_animated ? d->animated_index_count : 0) >= (1ull << 32))
        return fail(ctx, PT_ERR_UNSUPPORTED, "pt_scene_upload", "more than 2^32 vertices or indices");

    freeScene(ctx);
    std::vector<void *> &own = ctx->sceneAllocs;
    std::vector<void *> temp;
    auto freeTemp = [&]() {
        for (void *p : temp)
            cudaFree(p);
        temp.clear();
    };
    ScopedEvent ev0, ev1, ev2; // destroyed on every (error) path out of this function
    cudaEventRecord(ev0, ctx->stream);

#define PT_TRY(expr)                                                                                                  \
    do                                                                                                                \
    {                                                                                                                 \
        const pt_status st__ = (expr);                                                                                \
        if (st__ != PT_OK)                                                                                            \
        {                                                                                                             \
            freeTemp();                                                                                               \
            freeScene(ctx);                                                                                           \
            return st__;                                                                                              \
        }                                                                                                             \
    } while (0)

    // ---- host copy of the instance / model / mesh tables (pt_scene_update re-flattens from them) ----
    SceneTopology &topo = ctx->topo;
    topo.instances.assign(d->instances, d->instances + d->instance_count);
    topo.models.assign(d->models, d->models + d->model_count);
    topo.meshRecords.assign(d->mesh_records, d->mesh_records + d->mesh_record_count);
    topo.geometries.assign(d->geometries, d->geometries + d->geometry_count);
    topo.transforms.assign(d->transforms, d->transforms + 12 * (size_t)d->transform_count);
    topo.vertexCount = d->vertex_count;
    topo.indexCount = d->index_count;
    topo.materialCount[0] = d->mr_material_count;
    topo.materialCount[1] = d->sg_material_count;
    topo.materialCount[2] = d->phong_material_count;
    topo.geometryIsAnimated.clear();
    topo.animatedVertexCount = topo.animatedIndexCount = 0;
    topo.boneCount = 0;
    if (d->geometry_is_animated)
    {
        topo.geometryIsAnimated.assign(d->geometry_is_animated, d->geometry_is_animated + d->geometry_count);
        topo.animatedVertexCount = d->animated_vertex_count;
        topo.animatedIndexCount = d->animated_index_count;
        topo.boneCount = d->bone_count;
    }
    std::vector<MeshInstance> mis;
    bool hasAlpha = false;
    PT_TRY(flattenInstances(ctx, topo, mis, hasAlpha));
    const uint32_t n = mis.empty() ? 0u : mis.back().triOffset + mis.back().triCount;

    // ---- materials, lights, LUT, textures -------------------------------------------------
    DeviceScene &s = ctx->scene;
    {
        MaterialRaw *dm[3];
        const void *src[3] = { d->mr_materials, d->sg_materials, d->phong_materials };
        const uint32_t cnt[3] = { d->mr_material_count, d->sg_material_count, d->phong_material_count };
        for (int k = 0; k < 3; k++)
        {
            PT_TRY(devAlloc(ctx, &dm[k], cnt[k], own));
            if (cnt[k])
                PT_CUDA_CHECK(ctx, cudaMemcpyAsync(dm[k], src[k], (size_t)cnt[k] * 96, cudaMemcpyHostToDevice, ctx->stream));
            s.materials[k] = dm[k];
        }
        LightBlock &lb = ctx->hostLights;
        lb = LightBlock {};
        lb.count = d->point_light_count;
        lb.dirColor = make_float4(d->directional_light.color[0], d->directional_light.color[1], d->directional_light.color[2], 0);
        lb.dirDirection = make_float4(d->directional_light.direction[0], d->directional_light.direction[1],
                                      d->directional_light.direction[2], 0);
        if (d->point_light_count)
            std::memcpy(lb.point, d->point_lights, (size_t)d->point_light_count * 48);
        LightBlock *dl;
        PT_TRY(devAlloc(ctx, &dl, 1, own));
        PT_CUDA_CHECK(ctx, cudaMemcpyAsync(dl, &lb, sizeof(lb), cudaMemcpyHostToDevice, ctx->stream));
        PT_CUDA_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
        s.lights = dl;
        s.lut = ctx->dLut;
    }
    {
        // built-in 1x1 textures, slots 0-8 (PT/Renderer/Renderer.cpp:127-173; texel values
        // PT/Shaders/ShaderRendererTypes.incl:49-56; colour space per texture type).  Slot 8 is the
        // reference's "placeholder" shown while uploads are pending; uploads here are synchronous.
        static const uint32_t kDefaults[9] = { 0xffffffffu, 0xffff8080u, 0xffffffffu, 0xffffffffu, 0x00000000u,
                                               0xffffffffu, 0x00000000u, 0x00000000u, 0xffffffffu };
        static const bool kSrgb[9] = { true, false, false, false, true, true, false, false, true };
        // the six faces of a cube sky follow the scene's textures in the same table
        const uint32_t sceneSlots = PT_SCENE_TEXTURE_OFFSET + d->texture_count;
        if (d->skybox_cube)
            for (int f = 1; f < 6; f++)
                if (d->skybox_cube[f].width != d->skybox_cube[0].width || d->skybox_cube[f].height != d->skybox_cube[0].height ||
                    d->skybox_cube[f].format != d->skybox_cube[0].format)
                    return fail(ctx, PT_ERR_INVALID_ARGUMENT, "pt_scene_upload", "cube sky faces differ in size or format");
        ctx->hostTextures.resize(sceneSlots + (d->skybox_cube ? 6 : 0));
        ctx->textureBudgetCount = std::max(1u, d->texture_count); // TextureUploader.cpp:554: the budget is shared by the scene's textures
        s.skyCubeSlot = d->skybox_cube ? sceneSlots : 0;
        for (uint32_t i = 0; i < ctx->hostTextures.size(); i++)
        {
            const pt_texture_desc desc = i < PT_SCENE_TEXTURE_OFFSET ? defaultTexture(&kDefaults[i], kSrgb[i])
                                         : i < sceneSlots            ? d->textures[i - PT_SCENE_TEXTURE_OFFSET]
                                                                     : d->skybox_cube[i - sceneSlots];
            void *mem = nullptr;
            PT_TRY(createTexture(ctx, desc, ctx->hostTextures[i], &mem, i >= PT_SCENE_TEXTURE_OFFSET && i < sceneSlots));
            own.push_back(mem);
        }
        DevTexture *dt;
        PT_TRY(devAlloc(ctx, &dt, ctx->hostTextures.size(), own));
        PT_CUDA_CHECK(ctx, cudaMemcpyAsync(dt, ctx->hostTextures.data(), ctx->hostTextures.size() * sizeof(DevTexture),
                                           cudaMemcpyHostToDevice, ctx->stream));
        s.textures = dt;
        s.textureCount = (uint32_t)ctx->hostTextures.size();
        s.hasSky2D = 0;
        if (d->skybox_2d)
        {
            void *mem = nullptr;
            PT_TRY(createTexture(ctx, *d->skybox_2d, s.sky2D, &mem));
            own.push_back(mem);
            s.hasSky2D = 1;
        }
    }
    // material texture indices must address existing slots
    {
        auto checkIdx = [&](uint32_t idx) { return idx < PT_SCENE_TEXTURE_OFFSET + d->texture_count; };
        bool ok = true;
        for (uint32_t i = 0; i < d->mr_material_count; i++)
        {
            const pt_material_mr &m = d->mr_materials[i];
            ok &= checkIdx(m.emissive_idx) && checkIdx(m.color_idx) && checkIdx(m.normal_idx) && checkIdx(m.roughness_idx) &&
                  checkIdx(m.metallic_idx);
        }
        for (int k = 0; k < 2; k++)
        {
            const pt_material_sg *arr = k == 0 ? d->sg_materials : d->phong_materials;
            const uint32_t cnt = k == 0 ? d->sg_material_count : d->phong_material_count;
            for (uint32_t i = 0; i < cnt; i++)
                ok &= checkIdx(arr[i].emissive_idx) && checkIdx(arr[i].color_idx) && checkIdx(arr[i].normal_idx) &&
                      checkIdx(arr[i].specular_idx) && checkIdx(arr[i].glossiness_idx);
        }
        if (!ok)
        {
            freeTemp();
            freeScene(ctx);
            return fail(ctx, PT_ERR_INVALID_ARGUMENT, "pt_scene_upload", "material texture index out of range");
        }
    }

    // (s.triCount was set by buildAccel: the number of leaf entries = references)
    s.hasAlpha = hasAlpha ? 1u : 0u;
    s.maxAnisotropy = ctx->maxAnisotropy;
    // vertices and indices stay on the device: pt_scene_update re-bakes from them.  Skinned vertices and
    // animated indices follow the static ones in the same buffers.
    {
        float *dVertices;
        uint32_t *dIndices;
        const uint64_t av = topo.animatedVertexCount, ai = topo.animatedIndexCount;
        PT_TRY(devAlloc(ctx, &dVertices, (size_t)(d->vertex_count + av) * 14, own));
        PT_TRY(devAlloc(ctx, &dIndices, (size_t)(d->index_count + ai), own));
        if (d->vertex_count)
            PT_CUDA_CHECK(ctx, cudaMemcpyAsync(dVertices, d->vertices, (size_t)d->vertex_count * 56, cudaMemcpyHostToDevice, ctx->stream));
        if (d->index_count)
            PT_CUDA_CHECK(ctx, cudaMemcpyAsync(dIndices, d->indices, (size_t)d->index_count * 4, cudaMemcpyHostToDevice, ctx->stream));
        if (ai)
            PT_CUDA_CHECK(ctx, cudaMemcpyAsync(dIndices + d->index_count, d->animated_indices, (size_t)ai * 4, cudaMemcpyHostToDevice, ctx->stream));
        ctx->dVertices = dVertices;
        ctx->dIndices = dIndices;
        ctx->dAnimatedVertices = nullptr;
        ctx->dBones = nullptr;
        if (av)
        {
            float *dAnimated;
            PT_TRY(devAlloc(ctx, &dAnimated, (size_t)av * 22, own));
            PT_TRY(devAlloc(ctx, &ctx->dBones, (size_t)topo.boneCount * PT_BONE_STRIDE, own));
            PT_CUDA_CHECK(ctx, cudaMemcpyAsync(dAnimated, d->animated_vertices, (size_t)av * 88, cudaMemcpyHostToDevice, ctx->stream));
            ctx->dAnimatedVertices = dAnimated;
        }
        PT_CUDA_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
        if (av)
            PT_TRY(skinAnimatedVertices(ctx, d->bone_transforms));
    }
    cudaEventRecord(ev1, ctx->stream);
    PT_TRY(buildAccel(ctx, mis, n));
    cudaEventRecord(ev2, ctx->stream);
    PT_CUDA_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    PT_CUDA_CHECK(ctx, cudaGetLastError());
    freeTemp();
    cudaEventElapsedTime(&ctx->sceneUploadMs, ev0, ev2);
    cudaEventElapsedTime(&ctx->bvhBuildMs, ev1, ev2);
    ctx->hasScene = true;
    ctx->sceneUpdates = 0;
    return PT_OK;
#undef PT_TRY
}

// Scene::Update's per-frame outputs (PT/Scene.cpp:52-83: instance transforms, point-light positions,
// directional-light direction) applied to the uploaded scene.  The reference refits its BLASes and
// TLAS in place (AccelerationStructure::RecordUpdateCommands, AccelerationStructure.cpp:48-57); here
// the instances are re-baked and the BVH is REBUILT on the GPU — a full PLOC build of a few million
// triangles costs about as much as one sample per pixel, and a fresh tree keeps its quality however
// far the instances move.
pt_status updateScene(Context *ctx, const pt_scene_update_desc *d)
{
    if (!d)
        return fail(ctx, PT_ERR_INVALID_ARGUMENT, "pt_scene_update", "desc is NULL");
    if (!ctx->hasScene)
        return fail(ctx, PT_ERR_NO_SCENE, "pt_scene_update", "no scene uploaded");
    if (d->instance_transforms && d->instance_count != ctx->topo.instances.size())
        return fail(ctx, PT_ERR_INVALID_ARGUMENT, "pt_scene_update", "instance_count differs from the uploaded scene");
    if (d->point_lights && d->point_light_count > PT_MAX_LIGHT_COUNT)
        return fail(ctx, PT_ERR_INVALID_ARGUMENT, "pt_scene_update", "more than 64 point lights");
    if (d->bone_transforms && (d->bone_count != ctx->topo.boneCount || ctx->topo.animatedVertexCount == 0))
        return fail(ctx, PT_ERR_INVALID_ARGUMENT, "pt_scene_update", "bone_count differs from the uploaded scene");
    PT_CUDA_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    if (d->point_lights || d->directional_light)
    {
        LightBlock &lb = ctx->hostLights;
        if (d->point_lights)
        {
            lb.count = d->point_light_count;
            if (d->point_light_count)
                std::memcpy(lb.point, d->point_lights, (size_t)d->point_light_count * 48);
        }
        if (d->directional_light)
        {
            lb.dirColor = make_float4(d->directional_light->color[0], d->directional_light->color[1], d->directional_light->color[2], 0);
            lb.dirDirection = make_float4(d->directional_light->direction[0], d->directional_light->direction[1],
                                          d->directional_light->direction[2], 0);
        }
        PT_CUDA_CHECK(ctx, cudaMemcpyAsync(const_cast<LightBlock *>(ctx->scene.lights), &lb, sizeof(lb), cudaMemcpyHostToDevice, ctx->stream));
        PT_CUDA_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    }
    if (d->bone_transforms)
    {
        const pt_status st = skinAnimatedVertices(ctx, d->bone_transforms);
        if (st != PT_OK)
            return st;
    }
    if (d->instance_transforms || d->bone_transforms)
    {
        ctx->emittersValid = false; // the emitters' corners move with the geometry
        if (d->instance_transforms)
            for (uint32_t i = 0; i < d->instance_count; i++)
                std::memcpy(ctx->topo.instances[i].transform, d->instance_transforms + 12 * (size_t)i, 48);
        std::vector<MeshInstance> mis;
        bool hasAlpha = false;
        pt_status st = flattenInstances(ctx, ctx->topo, mis, hasAlpha);
        if (st != PT_OK)
            return st;
        const uint32_t n = mis.empty() ? 0u : mis.back().triOffset + mis.back().triCount;
        cudaEvent_t ev0, ev1;
        cudaEventCreate(&ev0);
        cudaEventCreate(&ev1);
        cudaEventRecord(ev0, ctx->stream);
        st = buildAccel(ctx, mis, n);
        cudaEventRecord(ev1, ctx->stream);
        cudaEventSynchronize(ev1);
        if (st == PT_OK)
            cudaEventElapsedTime(&ctx->bvhBuildMs, ev0, ev1);
        cudaEventDestroy(ev0);
        cudaEventDestroy(ev1);
        if (st != PT_OK)
        {
            freeScene(ctx); // the old tree is gone and the new one failed: nothing left to render
            return st;
        }
    }
    ctx->sceneUpdates++;
    return PT_OK;
}

} // namespace pt
