// shading.cuh — device functions of the path-tracing hot path (sm_100a).
//
// Semantics follow the reference's GLSL (citations: PT/ = Path-Tracing/ in the reference
// checkout); the code is restructured for the GPU: shared sub-expressions of the reflection
// lobes are evaluated once, the orthonormal tangent frame is inverted by transposition, all
// per-hit matrix work is replaced by data baked at scene upload.  RNG consumption order is kept
// exactly (SURVEY Appendix B) because the stream is threaded through every stage.
#pragma once
#include "scene.cuh"
#include "vecmath.cuh"

namespace pt
{

#define PT_PI 3.14159265359f // PT/Shaders/common.glsl:3

// ---------------------------------------------------------------------------------------------
// RNG — PT/Shaders/common.glsl:133-165
// ---------------------------------------------------------------------------------------------
PT_HD uint32_t jenkinsHash(uint32_t x)
{
    x += x << 10;
    x ^= x >> 6;
    x += x << 3;
    x ^= x >> 11;
    x += x << 15;
    return x;
}
// dot(uvec2 pixel, uvec2(1, resolution.x)) is an integer dot product
PT_HD uint32_t initRng(uint32_t px, uint32_t py, uint32_t resX, uint32_t frame)
{
    return jenkinsHash((px + py * resX) ^ jenkinsHash(frame));
}
PT_DEV float rnd(uint32_t &s)
{
    s ^= s << 13;
    s ^= s >> 17;
    s ^= s << 5;
    return __uint_as_float(0x3f800000u | (s >> 9)) - 1.0f;
}

// ---------------------------------------------------------------------------------------------
// sampling helpers — PT/Shaders/common.glsl:168-202
// ---------------------------------------------------------------------------------------------
PT_DEV vec2 sampleUniformDiskConcentric(vec2 u)
{
    const vec2 offset = V2(2.0f * u.x - 1.0f, 2.0f * u.y - 1.0f);
    if (offset.x == 0.0f && offset.y == 0.0f)
        return V2(0.0f, 0.0f);
    float r, theta;
    if (fabsf(offset.x) > fabsf(offset.y))
    {
        r = offset.x;
        theta = (PT_PI / 4) * (offset.y / offset.x);
    }
    else
    {
        r = offset.y;
        theta = PT_PI / 2 - (PT_PI / 4) * (offset.x / offset.y);
    }
    float s, c;
    sincosf(theta, &s, &c);
    return V2(r * c, r * s);
}
PT_DEV vec3 sampleCosineHemisphere(vec2 u)
{
    const vec2 d = sampleUniformDiskConcentric(u);
    return V3(d.x, d.y, sqrtf(1 - d.x * d.x - d.y * d.y));
}
// mat3(normalize(tangent), normalize(bitangent), normal)
PT_DEV mat3 computeTangentSpace(vec3 n)
{
    const vec3 t1 = cross(n, V3(1.0f, 0.0f, 0.0f));
    const vec3 t2 = cross(n, V3(0.0f, 1.0f, 0.0f));
    const vec3 tangent = length(t1) > length(t2) ? t1 : t2;
    const vec3 bitangent = cross(n, tangent);
    return mat3 { normalize(tangent), normalize(bitangent), n };
}

// ---------------------------------------------------------------------------------------------
// microfacet core — PT/Shaders/shading.glsl
// ---------------------------------------------------------------------------------------------
// :3-14 — note D <= 1 through max(denom, 1)
PT_DEV float GGXDistribution(vec3 H, float alpha)
{
    const float alpha2 = alpha * alpha;
    const float s = H.x * H.x / alpha2 + H.y * H.y / alpha2 + H.z * H.z;
    const float denom = PT_PI * alpha2 * (s * s);
    return 1.0f / fmaxf(denom, 1.0f);
}
// :16-27
PT_DEV float Lambda(vec3 V, float alpha)
{
    const float alpha2 = alpha * alpha;
    const float Vz2 = fabsf(V.z) * fabsf(V.z);
    return (sqrtf(1.0f + (alpha2 * (V.x * V.x) + alpha2 * (V.y * V.y)) / Vz2) - 1.0f) / 2.0f;
}
// :29-32
PT_DEV float GGXSmith(vec3 V, float alpha) { return 1.0f / (1.0f + Lambda(V, alpha)); }
// :34-48
PT_DEV float DielectricFresnel(float VdotH, float eta)
{
    const float cosThetaI = VdotH;
    const float sinThetaT2 = eta * eta * (1.0f - cosThetaI * cosThetaI);
    if (sinThetaT2 > 1.0f)
        return 1.0f;
    const float cosThetaT = sqrtf(fmaxf(1.0f - sinThetaT2, 0.0f));
    const float rs = (eta * cosThetaT - cosThetaI) / (eta * cosThetaT + cosThetaI);
    const float rp = (eta * cosThetaI - cosThetaT) / (eta * cosThetaI + cosThetaT);
    return (rs * rs + rp * rp) / 2.0f;
}
// :50-53 — x^5 by squaring
PT_DEV float SchlickFresnel(float VdotH)
{
    const float x = clampf(1.0f - VdotH, 0.0f, 1.0f);
    const float x2 = x * x;
    return x2 * x2 * x;
}
// :56-77
PT_DEV vec3 EvaluateReflection(vec3 V, vec3 L, vec3 F, float alpha, float &pdf)
{
    if (L.z < 0.00001f)
    {
        pdf = 0.0f;
        return V3(0.0f);
    }
    const vec3 H = normalize(V + L);
    const float VdotH = dot(V, H);
    const float D = GGXDistribution(H, alpha);
    const float Gv = GGXSmith(V, alpha);
    const float Gl = GGXSmith(L, alpha);
    const float G = Gv * Gl;
    const float Dv = (Gv * fmaxf(VdotH, 0.0f) * D) / V.z;
    pdf = Dv / (4.0f * VdotH);
    return ((D * G) * F) / (4.0f * V.z);
}
// :80-108
PT_DEV vec3 EvaluateRefraction(vec3 V, vec3 L, vec3 F, float alpha, float eta, float &pdf)
{
    if (L.z > -0.00001f)
    {
        pdf = 0.0f;
        return V3(0.0f);
    }
    vec3 H = normalize(eta * V + L);
    if (H.z < 0.0f)
        H = -H;
    const float VdotH = dot(V, H);
    const float LdotH = dot(L, H);
    const float D = GGXDistribution(H, alpha);
    const float Gv = GGXSmith(V, alpha);
    const float Gl = GGXSmith(L, alpha);
    const float G = Gv * Gl;
    const float Dv = (Gv * fabsf(VdotH) * D) / V.z;
    const float denominator = LdotH + eta * VdotH;
    const float jacobian = ((eta * eta) * fabsf(LdotH)) / (denominator * denominator);
    pdf = Dv * jacobian;
    return (fabsf(VdotH) / fabsf(V.z)) * ((D * G) * F) * jacobian;
}
// :111-129 (Heitz 2018 VNDF sampling)
PT_DEV vec3 SampleGGX(vec2 u, vec3 V, float alpha)
{
    const vec3 Vh = normalize(V3(alpha * V.x, alpha * V.y, fabsf(V.z)));
    const float lensq = Vh.x * Vh.x + Vh.y * Vh.y;
    const vec3 T1 = lensq > 0 ? V3(-Vh.y, Vh.x, 0) * (1.0f / sqrtf(lensq)) : V3(1, 0, 0);
    const vec3 T2 = cross(Vh, T1);
    const float r = sqrtf(u.x);
    const float phi = (2.0f * PT_PI) * u.y;
    float sp, cp;
    sincosf(phi, &sp, &cp);
    const float t1 = r * cp;
    float t2 = r * sp;
    const float s = 0.5f * (1.0f + Vh.z);
    t2 = (1.0f - s) * sqrtf(1.0f - t1 * t1) + s * t2;
    const vec3 Nh = t1 * T1 + t2 * T2 + sqrtf(fmaxf(0.0f, 1.0f - t1 * t1 - t2 * t2)) * Vh;
    return normalize(V3(alpha * Nh.x, alpha * Nh.y, fmaxf(0.0f, Nh.z)));
}

// ---------------------------------------------------------------------------------------------
// BSDF — PT/Shaders/bsdf.glsl
// ---------------------------------------------------------------------------------------------
// Shaders::MaterialSample, PT/Shaders/ShaderRendererTypes.incl:129-140
struct MaterialSample
{
    vec3 EmissiveColor;
    vec3 Color;
    vec3 Normal;
    float Roughness;
    float Metalness;
    float Transmission;
    float Eta;
    vec3 AttenuationColor;
    float AttenuationDistance;
};

struct LobePdfs
{
    float Diffuse, Glossy, Metallic, Transmissive;
};
// :62-70
PT_DEV LobePdfs sampleLobePdfs(float metalness, float transmission, float F)
{
    LobePdfs p;
    p.Diffuse = (1.0f - metalness) * (1.0f - F) * (1.0f - transmission);
    p.Glossy = (1.0f - metalness) * F;
    p.Metallic = metalness;
    p.Transmissive = (1.0f - metalness) * (1.0f - F) * transmission;
    return p;
}

// :72-103.  The glossy (:22-25) and metallic (:32-37) lobes share H, D, G and the pdf; they are
// evaluated once and weighted separately, in the reference's summation order.
PT_DEV vec3 evaluateBSDF(const MaterialSample &m, vec3 V, vec3 L, float &outPdf)
{
    const bool isReflection = L.z > 0.0f;
    const float alpha = m.Roughness * m.Roughness;
    if (isReflection)
    {
        const vec3 H = normalize(V + L);
        const float VdotH = dot(V, H);
        const float FD = DielectricFresnel(fabsf(VdotH), m.Eta);
        const LobePdfs w = sampleLobePdfs(m.Metalness, m.Transmission, FD);

        // diffuse :11-15
        float pdf = L.z * 1.0f / PT_PI;
        vec3 bsdf = (L.z * m.Color / PT_PI) * w.Diffuse;
        outPdf = 0.0f + pdf * w.Diffuse;

        // EvaluateReflection shared part
        vec3 glossy = V3(0.0f), metallic = V3(0.0f);
        float pdfR = 0.0f;
        if (!(L.z < 0.00001f))
        {
            const float D = GGXDistribution(H, alpha);
            const float Gv = GGXSmith(V, alpha);
            const float Gl = GGXSmith(L, alpha);
            const float DG = D * (Gv * Gl);
            const float Dv = (Gv * fmaxf(VdotH, 0.0f) * D) / V.z;
            pdfR = Dv / (4.0f * VdotH);
            const float den = 4.0f * V.z;
            glossy = V3(DG / den); // F = vec3(1): (D*G*1) / (4 V.z)
            const vec3 F0 = mix(m.Color, V3(1.0f), SchlickFresnel(VdotH));
            metallic = (DG * F0) / den;
        }
        bsdf += glossy * w.Glossy;
        outPdf += pdfR * w.Glossy;
        bsdf += metallic * w.Metallic;
        outPdf += pdfR * w.Metallic;
        return bsdf;
    }
    const vec3 H = normalize(m.Eta * V + L);
    const float FD = DielectricFresnel(fabsf(dot(V, H)), m.Eta);
    const LobePdfs w = sampleLobePdfs(m.Metalness, m.Transmission, FD);
    float pdf;
    const vec3 btdf = EvaluateRefraction(V, L, m.Color, alpha, m.Eta, pdf); // :44-47
    outPdf = 0.0f + pdf * w.Transmissive;
    return btdf * w.Transmissive;
}

struct BSDFSample
{
    vec3 Direction;
    float Pdf;
    vec3 Color;
};

// :105-132 — consumes 3, 4, 5 or 7 random numbers depending on the lobe taken
PT_DEV BSDFSample sampleBSDF(const MaterialSample &m, vec3 V, uint32_t &rng)
{
    const float alpha = m.Roughness * m.Roughness;
    const float u0 = rnd(rng);
    const float u1 = rnd(rng);
    const vec3 H = SampleGGX(V2(u0, u1), V, alpha);
    const float FD = DielectricFresnel(fabsf(dot(V, H)), m.Eta);
    vec3 L;
    if (rnd(rng) < m.Metalness)
        L = normalize(reflect(-V, H));
    else if (rnd(rng) < FD)
        L = normalize(reflect(-V, H));
    else if (rnd(rng) < m.Transmission)
        L = normalize(refract(-V, H, m.Eta));
    else
    {
        const float d0 = rnd(rng);
        const float d1 = rnd(rng);
        L = sampleCosineHemisphere(V2(d0, d1));
    }
    BSDFSample r;
    r.Direction = L;
    r.Color = evaluateBSDF(m, V, L, r.Pdf);
    return r;
}

// ---------------------------------------------------------------------------------------------
// ray origins — PT/Shaders/ray.glsl:93-131
// ---------------------------------------------------------------------------------------------
PT_DEV float offsetAxis(float o, float n)
{
    const int32_t of_i = (int32_t)(256.0f * n);
    const float p_i = __int_as_float(__float_as_int(o) + ((o < 0) ? -of_i : of_i));
    return (fabsf(o) < (1.0f / 32.0f)) ? o + (1.0f / 65536.0f) * n : p_i;
}
// Waechter & Binder
PT_DEV vec3 offsetRayOriginSelfIntersection(vec3 origin, vec3 normal)
{
    return V3(offsetAxis(origin.x, normal.x), offsetAxis(origin.y, normal.y), offsetAxis(origin.z, normal.z));
}
// Hanika: p, vertex positions and (unit) vertex normals in world space
PT_DEV vec3 offsetRayOriginShadowTerminator(vec3 p, vec3 p0, vec3 p1, vec3 p2, vec3 n0, vec3 n1, vec3 n2, vec3 bary,
                                            bool isRefracted)
{
    vec3 tmpu = p - p0, tmpv = p - p1, tmpw = p - p2;
    if (isRefracted)
    {
        n0 = -n0;
        n1 = -n1;
        n2 = -n2;
    }
    const float dotu = fminf(0.0f, dot(tmpu, n0));
    const float dotv = fminf(0.0f, dot(tmpv, n1));
    const float dotw = fminf(0.0f, dot(tmpw, n2));
    tmpu -= dotu * n0;
    tmpv -= dotv * n1;
    tmpw -= dotw * n2;
    return p + bary.x * tmpu + bary.y * tmpv + bary.z * tmpw;
}

// ---------------------------------------------------------------------------------------------
// camera — PT/Shaders/ray.glsl:16-90
// ---------------------------------------------------------------------------------------------
struct CameraMatrices
{
    float view[16]; // ViewInverse, column-major
    float proj[16]; // ProjInverse
};
PT_DEV vec3 mulPoint(const float *m, float x, float y, float z, float w)
{
    // (M * vec4).xyz summed pairwise, (c0*x + c1*y) + (c2*z + c3*w), as the reference's vendored glm (and with
    // it the oracle and the compiled-GLSL reference) evaluates mat4 * vec4 (glm/detail/type_mat4x4.inl)
    return V3((m[0] * x + m[4] * y) + (m[8] * z + m[12] * w), (m[1] * x + m[5] * y) + (m[9] * z + m[13] * w),
              (m[2] * x + m[6] * y) + (m[10] * z + m[14] * w));
}
struct PrimaryRays
{
    vec3 origin, direction, rxDirection, ryDirection; // rx/ry share the origin
};
PT_DEV PrimaryRays constructPrimaryRay(float px, float py, float resX, float resY, const CameraMatrices &cam, vec2 u,
                                       vec2 u2, float lensRadius, float focalDistance)
{
    const float cx = px + u.x, cy = py + u.y;
    const float dx = cx / resX * 2.0f - 1.0f, dy = cy / resY * 2.0f - 1.0f;
    const float dxo = (cx + 1.0f) / resX * 2.0f - 1.0f, dyo = (cy + 1.0f) / resY * 2.0f - 1.0f;
    const vec3 target = mulPoint(cam.proj, dx, dy, 1, 1);
    const vec3 targetX = mulPoint(cam.proj, dxo, dy, 1, 1);
    const vec3 targetY = mulPoint(cam.proj, dx, dyo, 1, 1);
    PrimaryRays r;
    if (lensRadius > 0)
    {
        const vec2 disk = sampleUniformDiskConcentric(u2);
        const vec3 oc = V3(lensRadius * disk.x, lensRadius * disk.y, 0);
        r.origin = mulPoint(cam.view, oc.x, oc.y, oc.z, 1);
        const vec3 d0 = normalize((focalDistance / target.z) * target - oc);
        const vec3 d1 = normalize((focalDistance / targetX.z) * targetX - oc);
        const vec3 d2 = normalize((focalDistance / targetY.z) * targetY - oc);
        r.direction = mulPoint(cam.view, d0.x, d0.y, d0.z, 0);
        r.rxDirection = mulPoint(cam.view, d1.x, d1.y, d1.z, 0);
        r.ryDirection = mulPoint(cam.view, d2.x, d2.y, d2.z, 0);
    }
    else
    {
        r.origin = mulPoint(cam.view, 0, 0, 0, 1);
        const vec3 d0 = normalize(target), d1 = normalize(targetX), d2 = normalize(targetY);
        r.direction = mulPoint(cam.view, d0.x, d0.y, d0.z, 0);
        r.rxDirection = mulPoint(cam.view, d1.x, d1.y, d1.z, 0);
        r.ryDirection = mulPoint(cam.view, d2.x, d2.y, d2.z, 0);
    }
    return r;
}

// ---------------------------------------------------------------------------------------------
// ray differentials — PT/Shaders/tracing.glsl
// ---------------------------------------------------------------------------------------------
// :44-50
PT_DEV float differenceOfProducts(float a, float b, float c, float d)
{
    const float cd = c * d;
    const float dop = fmaf(a, b, -cd);
    const float err = fmaf(-c, d, cd);
    return dop + err;
}
PT_DEV float clampDerivative(float v) { return isinf(v) ? 0.0f : clampf(v, -1e8f, 1e8f); }
// :53-78 -> (dudx, dvdx, dudy, dvdy)
PT_DEV float4 computeDerivatives(vec3 dpdx, vec3 dpdy, vec3 dpdu, vec3 dpdv)
{
    const float ata00 = dot(dpdu, dpdu), ata01 = dot(dpdu, dpdv), ata11 = dot(dpdv, dpdv);
    float invDet = 1 / differenceOfProducts(ata00, ata11, ata01, ata01);
    invDet = isinf(invDet) ? 0.0f : invDet;
    const float atb0x = dot(dpdu, dpdx), atb1x = dot(dpdv, dpdx);
    const float atb0y = dot(dpdu, dpdy), atb1y = dot(dpdv, dpdy);
    const float dudx = differenceOfProducts(ata11, atb0x, ata01, atb1x) * invDet;
    const float dvdx = differenceOfProducts(ata00, atb1x, ata01, atb0x) * invDet;
    const float dudy = differenceOfProducts(ata11, atb0y, ata01, atb1y) * invDet;
    const float dvdy = differenceOfProducts(ata00, atb1y, ata01, atb0y) * invDet;
    return make_float4(clampDerivative(dudx), clampDerivative(dvdx), clampDerivative(dudy), clampDerivative(dvdy));
}

// :2-28 with e1 = p1 - p0, e2 = p2 - p0 (world space), en = normal differences, duv = uv differences
PT_DEV void computeDpnDuv(vec3 e1, vec3 e2, vec3 en1, vec3 en2, vec2 duv1, vec2 duv2, vec3 tangent, vec3 bitangent, vec3 &dpdu,
                          vec3 &dpdv, vec3 &dndu, vec3 &dndv)
{
    const float det = duv1.x * duv2.y - duv2.x * duv1.y;
    if (fabsf(det) < 1e-8f)
    {
        dpdu = tangent;
        dpdv = bitangent;
        dndu = V3(0.0f);
        dndv = V3(0.0f);
    }
    else
    {
        const float invDet = 1.0f / det;
        dpdu = (duv2.y * e1 - duv1.y * e2) * invDet;
        dpdv = (-duv2.x * e1 + duv1.x * e2) * invDet;
        dndu = (duv2.y * en1 - duv1.y * en2) * invDet;
        dndv = (-duv2.x * en1 + duv1.x * en2) * invDet;
    }
}
// :31-41
PT_DEV void computeDpDxy(vec3 p, vec3 rxOrigin, vec3 rxDirection, vec3 ryOrigin, vec3 ryDirection, vec3 n, vec3 &dpdx, vec3 &dpdy)
{
    const float d = -dot(n, p);
    const float tx = (-dot(n, rxOrigin) - d) / dot(n, rxDirection);
    const float ty = (-dot(n, ryOrigin) - d) / dot(n, ryDirection);
    dpdx = (rxOrigin + tx * rxDirection) - p;
    dpdy = (ryOrigin + ty * ryDirection) - p;
}

struct RayDifferentials
{
    vec3 rxOrigin, rxDirection, ryOrigin, ryDirection;
};

// :81-108 and :111-148; `refracted` selects the transmission formulas
// (dndx, dndy) = dndu * derivatives.xz + dndv * derivatives.yw, the first two statements of the GLSL function, are
// the caller's: the wavefront computes them before the material fetch, where dndu / dndv / derivatives die
PT_DEV void propagateDifferentials(vec3 n, vec3 p, vec3 viewDir, vec3 newDir, vec3 dndx, vec3 dndy, float eta, bool refracted,
                                   RayDifferentials &rd)
{
    const float d = -dot(n, p);
    const float tx = (-dot(n, rd.rxOrigin) - d) / dot(n, rd.rxDirection);
    const vec3 px = rd.rxOrigin + tx * rd.rxDirection;
    const float ty = (-dot(n, rd.ryOrigin) - d) / dot(n, rd.ryDirection);
    const vec3 py = rd.ryOrigin + ty * rd.ryDirection;
    const vec3 dwodx = -rd.rxDirection - viewDir;
    const vec3 dwody = -rd.ryDirection - viewDir;
    rd.rxOrigin = px;
    rd.ryOrigin = py;
    if (!refracted)
    {
        const float dwoDotn_dx = dot(dwodx, n) + dot(viewDir, dndx);
        const float dwoDotn_dy = dot(dwody, n) + dot(viewDir, dndy);
        const float vn = dot(viewDir, n);
        rd.rxDirection = normalize(newDir - dwodx + 2 * (vn * dndx + dwoDotn_dx * n));
        rd.ryDirection = normalize(newDir - dwody + 2 * (vn * dndy + dwoDotn_dy * n));
        return;
    }
    if (dot(viewDir, n) < 0.0f)
    {
        n = -n;
        dndx = -dndx;
        dndy = -dndy;
    }
    const float dwoDotn_dx = dot(dwodx, n) + dot(viewDir, dndx);
    const float dwoDotn_dy = dot(dwody, n) + dot(viewDir, dndy);
    const float vn = dot(viewDir, n), rn = dot(newDir, n);
    const float mu = vn / eta - fabsf(rn);
    const float k = 1.0f / eta + 1.0f / (eta * eta) * vn / rn;
    const float dmudx = dwoDotn_dx * k;
    const float dmudy = dwoDotn_dy * k;
    rd.rxDirection = normalize(newDir - eta * dwodx + (mu * dndx + dmudx * n));
    rd.ryDirection = normalize(newDir - eta * dwody + (mu * dndy + dmudy * n));
}

PT_DEV void propagateDifferentials(float4 derivatives, vec3 n, vec3 p, vec3 viewDir, vec3 newDir, vec3 dndu, vec3 dndv,
                                   float eta, bool refracted, RayDifferentials &rd)
{
    const vec3 dndx = dndu * derivatives.x + dndv * derivatives.y;
    const vec3 dndy = dndu * derivatives.z + dndv * derivatives.w;
    propagateDifferentials(n, p, viewDir, newDir, dndx, dndy, eta, refracted, rd);
}

// common.glsl:17-20
PT_DEV vec3 hdrToLdr(vec3 rgb) { return rgb / (1.0f + maxComponent(rgb)); }

// material.glsl:55-60
PT_DEV vec3 reconstructNormalFromXY(float4 t)
{
    const float x = 2.0f * t.x - 1.0f, y = 2.0f * t.y - 1.0f;
    return V3(x, y, sqrtf(fmaxf(1 - x * x - y * y, 0.0f)));
}

// ---------------------------------------------------------------------------------------------
// sampling.glsl:25-56
// ---------------------------------------------------------------------------------------------
struct LightSample
{
    vec3 Direction;
    float Distance;
    vec3 Color;
    float Attenuation;
};

PT_DEV LightSample sampleLight(const LightBlock *lb, vec3 u, vec3 position, float &pdf)
{
    const uint32_t count = __ldg(&lb->count);
    const uint32_t lightIndex = (uint32_t)(u.x * (float)(count + 1));
    pdf = 1.0f / (float)(count + 1);
    const vec2 dp = sampleUniformDiskConcentric(V2(u.y, u.z));
    LightSample r;
    if (lightIndex >= count)
    {
        const vec3 diskPoint = V3(dp.x, dp.y, 0.0f) * 0.001f;
        const vec3 direction = normalize(V3(__ldg(&lb->dirDirection)));
        r.Direction = normalize(direction + mul(computeTangentSpace(direction), diskPoint));
        r.Color = V3(__ldg(&lb->dirColor));
        r.Distance = 100000.0f;
        r.Attenuation = 1.0f;
        return r;
    }
    const float4 lc = __ldg(&lb->point[lightIndex * 3]), lp = __ldg(&lb->point[lightIndex * 3 + 1]);
    const float4 la = __ldg(&lb->point[lightIndex * 3 + 2]);
    const vec3 diskPoint = V3(dp.x, dp.y, 0.0f) * 0.1f;
    const vec3 direction = normalize(position - V3(lp));
    const vec3 newPosition = V3(lp) + mul(computeTangentSpace(direction), diskPoint);
    r.Distance = length(position - newPosition);
    r.Direction = normalize(position - newPosition);
    r.Color = V3(lc);
    const float attenuation = 1.0f / (la.x + r.Distance * la.y + r.Distance * r.Distance * la.z);
    r.Attenuation = clampf(attenuation, 0.0f, 1.0f);
    return r;
}

// ---------------------------------------------------------------------------------------------
// emissive-triangle light sampling (PT_LIGHT_SAMPLING_EMISSIVE_MIS, DESIGN.md §3g) — an extension, no GLSL
// counterpart; tests/emissive_oracle.cpp defines the same functions
// ---------------------------------------------------------------------------------------------
// The emissive colour x intensity (q0) and emissive texture slot of a material; false when it cannot emit: intensity 0, or
// a zero colour with one of the black built-in 1x1 textures (slots 4, 6, 7)
PT_DEV bool emissiveSource(const DeviceScene &s, uint32_t materialId, float4 &q0, uint32_t &slot)
{
    const uint32_t type = materialId & 0xffu, index = materialId >> 8;
    if (type > 2)
        return false;
    const MaterialRaw *m = (type == 0 ? s.materials[0] : type == 1 ? s.materials[1] : s.materials[2]) + index;
    q0 = __ldg(&m->q[0]);
    const float4 q4 = __ldg(&m->q[4]);
    slot = __float_as_uint(type == 0 ? q4.w : q4.z);
    const bool blackTexture = slot == 4 || slot == 6 || slot == 7;
    return q0.w > 0.0f && (q0.x != 0.0f || q0.y != 0.0f || q0.z != 0.0f || !blackTexture);
}

// w = a^2 / (a^2 + b^2) for pdfs a, b >= 0: finite and in [0, 1] for every input, zero and infinite pdfs included
PT_DEV float powerHeuristic(float a, float b)
{
    if (!(a > 0.0f))
        return 0.0f;
    if (!(b > 0.0f))
        return 1.0f;
    if (isinf(a))
        return isinf(b) ? 0.5f : 1.0f;
    const float r = b / a;
    return 1.0f / (1.0f + r * r);
}

PT_DEV uint32_t xorshift(uint32_t &s)
{
    s ^= s << 13;
    s ^= s >> 17;
    s ^= s << 5;
    return s;
}

// the secondary stream of a light sample: a hash of the main stream's state, which is not advanced by it
PT_DEV uint32_t lightSampleRng(uint32_t rng) { return jenkinsHash(rng ^ 0x68bc21ebu); }


} // namespace pt
