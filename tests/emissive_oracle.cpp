/* emissive_oracle.cpp — the CPU reference of the emissive-MIS light sampling (PT_LIGHT_SAMPLING_EMISSIVE_MIS,
 * DESIGN.md section 3g): an extension mode with no GLSL counterpart, test infrastructure only.
 *
 * It extends the oracle without changing it: this translation unit includes oracle/pt_oracle.cpp, so the scene,
 * traversal, material, BSDF and sampler code are the oracle's own, and adds the emitter table and a raygen /
 * closest-hit pair with the emitter branch of the light sample and the MIS weight of emission found by BSDF sampling.
 * The reference mode is the oracle's pto_render of the same library.  The definitions are those of
 * path-tracing_b200/csrc/emitters.cu and k_shade_emissive; the emitter table is equal entry for entry. */
#include "../oracle/pt_oracle.cpp"

namespace
{

struct EmitterTable
{
    std::vector<uint32_t> emitterIds, emitterWeights; /* flat ids, integer weights */
    std::vector<uint32_t> aliasThreshold, aliasIndex;
    std::vector<float> emitterPdf;  /* P(select) / area of emitter k */
    std::vector<float> pdfOverArea; /* the same by flat id, 0 for triangles that are never sampled */
    float pEmitter = 0.0f;          /* emitter-branch probability; 0 = no emitters, the reference mode */
};

/* emissive colour, intensity and texture slot of a material; false when it cannot emit */
bool emissiveSource(const pto_scene &s, uint32_t materialId, vec3 &color, float &intensity, uint32_t &slot)
{
    uint32_t type;
    const uint32_t index = unpackMaterialId(materialId, type);
    const float *c;
    if (type == PT_MATERIAL_METALLIC_ROUGHNESS)
        c = s.mr[index].emissive_color, intensity = s.mr[index].emissive_intensity, slot = s.mr[index].emissive_idx;
    else if (type == PT_MATERIAL_SPECULAR_GLOSSINESS)
        c = s.sg[index].emissive_color, intensity = s.sg[index].emissive_intensity, slot = s.sg[index].emissive_idx;
    else if (type == PT_MATERIAL_PHONG)
        c = s.phong[index].emissive_color, intensity = s.phong[index].emissive_intensity, slot = s.phong[index].emissive_idx;
    else
        return false;
    color = V3(c[0], c[1], c[2]);
    const bool blackTexture = slot == 4 || slot == 6 || slot == 7;
    return intensity > 0.0f && (c[0] != 0.0f || c[1] != 0.0f || c[2] != 0.0f || !blackTexture);
}

void triangleUvs(const pto_scene &s, const FlatTri &ft, vec2 uv[3])
{
    const pt_geometry &g = s.geometries[meshRecordOf(s, ft).geometry_index];
    for (uint32_t k = 0; k < 3; k++)
        uv[k] = getVertex(s, g, ft.primitive * 3 + k).TexCoords;
}

/* Emitter set, integer weights and the alias table.  The arithmetic is spelled out operation by operation so that the
 * powers, and with them the table, are bit-identical to the GPU's. */
void buildEmitterTable(const pto_scene &s, EmitterTable &tab)
{
    tab.emitterIds.clear();
    std::vector<float> power, area;
    for (uint32_t f = 0; f < (uint32_t)s.tris.size(); f++)
    {
        const FlatTri &ft = s.tris[f];
        vec3 color;
        float intensity;
        uint32_t slot;
        if (!ft.opaque || !emissiveSource(s, meshRecordOf(s, ft).material_id, color, intensity, slot))
            continue;
        const vec3 a = ft.p1 - ft.p0, b = ft.p2 - ft.p0;
        const float cx = a.y * b.z - b.y * a.z, cy = a.z * b.x - b.z * a.x, cz = a.x * b.y - b.x * a.y;
        const float ar = 0.5f * std::sqrt(cx * cx + cy * cy + cz * cz);
        vec2 uv[3];
        triangleUvs(s, ft, uv);
        const float u = (uv[0].x + uv[1].x + uv[2].x) / 3.0f, v = (uv[0].y + uv[1].y + uv[2].y) / 3.0f;
        const float du = std::fmax(uv[0].x, std::fmax(uv[1].x, uv[2].x)) - std::fmin(uv[0].x, std::fmin(uv[1].x, uv[2].x));
        const float dv = std::fmax(uv[0].y, std::fmax(uv[1].y, uv[2].y)) - std::fmin(uv[0].y, std::fmin(uv[1].y, uv[2].y));
        const vec4 t = textureGrad(s.textures[slot], V2(u, v), V2(du, 0.0f), V2(0.0f, dv), nullptr, s.maxAnisotropy);
        const float ex = (t.x + color.x) * intensity, ey = (t.y + color.y) * intensity, ez = (t.z + color.z) * intensity;
        const float luminance = 0.2126f * ex + 0.7152f * ey + 0.0722f * ez;
        const float p = ar * std::fmax(luminance, 0.0f);
        if (std::isfinite(p) && p > 0.0f)
        {
            tab.emitterIds.push_back(f);
            power.push_back(p);
            area.push_back(ar);
        }
    }
    /* w = max(1, rint(power / maxPower * 2^24)); Vose's pairing, work lists in index order used as stacks */
    const size_t n = power.size();
    float maxPower = 0.0f;
    for (float p : power)
        maxPower = std::max(maxPower, p);
    tab.emitterWeights.assign(n, 0);
    tab.aliasThreshold.assign(n, 0);
    tab.aliasIndex.assign(n, 0);
    uint64_t W = 0;
    for (size_t k = 0; k < n; k++)
    {
        tab.emitterWeights[k] = std::max<uint32_t>(1u, (uint32_t)std::rint((double)power[k] / (double)maxPower * 16777216.0));
        W += tab.emitterWeights[k];
    }
    std::vector<uint64_t> share(n);
    std::vector<uint32_t> small, large;
    for (size_t k = 0; k < n; k++)
    {
        share[k] = (uint64_t)tab.emitterWeights[k] * n;
        (share[k] < W ? small : large).push_back((uint32_t)k);
    }
    while (!small.empty() && !large.empty())
    {
        const uint32_t l = small.back(), g = large.back();
        small.pop_back();
        tab.aliasThreshold[l] = (uint32_t)(((unsigned __int128)share[l] << 32) / W);
        tab.aliasIndex[l] = g;
        share[g] -= W - share[l];
        if (share[g] < W)
        {
            large.pop_back();
            small.push_back(g);
        }
    }
    for (const std::vector<uint32_t> *rest : { &small, &large })
        for (uint32_t k : *rest)
        {
            tab.aliasThreshold[k] = 0xffffffffu;
            tab.aliasIndex[k] = k;
        }
    tab.emitterPdf.assign(n, 0.0f);
    tab.pdfOverArea.assign(n ? s.tris.size() : 0, 0.0f);
    for (size_t k = 0; k < n; k++)
    {
        tab.emitterPdf[k] = (float)((double)tab.emitterWeights[k] / (double)W / (double)area[k]);
        tab.pdfOverArea[tab.emitterIds[k]] = tab.emitterPdf[k];
    }
    /* the emitter branch: never without emitters, always when no analytic light can contribute, else half the samples */
    const bool analytic = !s.pointLights.empty() || s.directional.color[0] != 0.0f || s.directional.color[1] != 0.0f ||
                          s.directional.color[2] != 0.0f;
    tab.pEmitter = n == 0 ? 0.0f : analytic ? 0.5f : 1.0f;
}

/* w = a^2 / (a^2 + b^2), finite and in [0, 1] for every input */
float powerHeuristic(float a, float b)
{
    if (!(a > 0.0f))
        return 0.0f;
    if (!(b > 0.0f))
        return 1.0f;
    if (std::isinf(a))
        return std::isinf(b) ? 0.5f : 1.0f;
    const float r = b / a;
    return 1.0f / (1.0f + r * r);
}

bool emissiveMode(const EmitterTable &t) { return t.pEmitter > 0.0f; }

/* a uniform point on emitter k seen from `position`, in sampleLight's form; pdf in solid angle (0: cannot be seen) */
LightSample sampleEmitter(const pto_scene &s, const EmitterTable &t, uint32_t k, float r1, float r2, vec3 position, float &pdf)
{
    const FlatTri &ft = s.tris[t.emitterIds[k]];
    const float su = std::sqrt(r1);
    const float b0 = 1.0f - su, b1 = su * (1.0f - r2), b2 = su * r2;
    const vec3 y = ft.p0 * b0 + ft.p1 * b1 + ft.p2 * b2;
    vec2 uv[3];
    triangleUvs(s, ft, uv);
    const vec2 texCoords = V2(uv[0].x * b0 + uv[1].x * b1 + uv[2].x * b2, uv[0].y * b0 + uv[1].y * b1 + uv[2].y * b2);
    const vec3 ng = normalize(cross(ft.p1 - ft.p0, ft.p2 - ft.p0));
    const vec3 target = offsetRayOriginSelfIntersection(y, dot(ng, position - y) >= 0.0f ? ng : -ng);
    LightSample r;
    r.Distance = length(position - target);
    r.Direction = normalize(position - target);
    vec3 color;
    float intensity;
    uint32_t slot;
    emissiveSource(s, meshRecordOf(s, ft).material_id, color, intensity, slot);
    r.Color = (xyz(textureLod0(s.textures[slot], texCoords)) + color) * intensity;
    r.Attenuation = 1.0f;
    const float cosLight = std::fabs(dot(ng, r.Direction));
    pdf = t.pEmitter * t.emitterPdf[k] * (r.Distance * r.Distance) / cosLight;
    if (!(pdf > 0.0f) || std::isinf(pdf))
        pdf = 0.0f;
    return r;
}

/* closestHitShader (PT/Shaders/closestHit.rchit:52-161) with the emitter branch of the light sample and the MIS weight
 * of the emission; bounce = this hit's bounce, emitterSample = the light sample is an emitter's */
void closestHitEmissive(const pto_scene &s, const EmitterTable &em, const pt_render_params &p, const HitInfo &hit,
                        vec3 rayOriginWorld, vec3 rayDirWorld, Payload &payload, uint32_t bounce, uint32_t &emitterSample,
                        Counters &c)
{
    const FlatTri &ft = s.tris[hit.tri];
    const pt_instance &inst = s.instances[ft.instance];
    const pt_mesh_record &sbt = meshRecordOf(s, ft);
    const pt_geometry &geom = s.geometries[sbt.geometry_index];
    const mat3x4 objectToWorld = objectToWorld3x4(inst);
    const uint32_t primitiveID = ft.primitive;
    const float rayTmax = hit.t;

    const vec3 barycentricCoords = computeBarycentricCoords(V2(hit.b1, hit.b2));

    Vertex v0 = getVertex(s, geom, primitiveID * 3);
    Vertex v1 = getVertex(s, geom, primitiveID * 3 + 1);
    Vertex v2 = getVertex(s, geom, primitiveID * 3 + 2);
    const Vertex originalVertex = interpolate(v0, v1, v2, barycentricCoords);
    Vertex vertex = transformVertex(s, originalVertex, sbt.transform_index, objectToWorld);

    v0 = transformVertex(s, v0, sbt.transform_index, objectToWorld);
    v1 = transformVertex(s, v1, sbt.transform_index, objectToWorld);
    v2 = transformVertex(s, v2, sbt.transform_index, objectToWorld);

    vec3 edge1 = v1.Position - v0.Position;
    vec3 edge2 = v2.Position - v0.Position;
    vec3 geometricNormal = normalize(cross(edge1, edge2));

    const bool isHitFromInside = dot(geometricNormal, rayDirWorld) > 0.0f;
    if (isHitFromInside)
    {
        geometricNormal *= -1.0f;
        vertex.Normal *= -1.0f;
        vertex.Tangent *= -1.0f;
        vertex.Bitangent *= -1.0f;
    }

    const vec3 viewDir = rayDirWorld;
    (void)rayOriginWorld;

    vec3 dpdu, dpdv, dndu, dndv;
    computeDpnDuv(v0, v1, v2, vertex, dpdu, dpdv, dndu, dndv);

    vec3 rxOrigin = xyz(payload.RayDifferentials0);
    vec3 rxDirection = V3(payload.RayDifferentials0.w, payload.RayDifferentials1.x, payload.RayDifferentials1.y);
    vec3 ryOrigin = V3(payload.RayDifferentials1.z, payload.RayDifferentials1.w, payload.RayDifferentials2.x);
    vec3 ryDirection = V3(payload.RayDifferentials2.y, payload.RayDifferentials2.z, payload.RayDifferentials2.w);

    vec3 dpdx, dpdy;
    computeDpDxy(vertex.Position, rxOrigin, rxDirection, ryOrigin, ryDirection, vertex.Normal, dpdx, dpdy);

    const vec4 derivatives = computeDerivatives(dpdx, dpdy, dpdu, dpdv);

    const bool flipYNormal = (p.hit_flags & PT_HIT_FLAGS_DX_NORMAL_TEXTURES) != 0;
    MaterialSample material =
        sampleMaterial(s, sbt.material_id, vertex.TexCoords, derivatives, isHitFromInside, flipYNormal, c);
    /* MIS weight of emission found by BSDF sampling (payload.Pdf is still the previous bounce's) */
    float emissionWeight = 1.0f;
    if (emissiveMode(em) && bounce != 0 && em.pdfOverArea[hit.tri] > 0.0f)
    {
        const vec3 g = normalize(cross(ft.p1 - ft.p0, ft.p2 - ft.p0));
        const float cosLight = std::fabs(dot(g, rayDirWorld));
        const float pdfLight = em.pEmitter * em.pdfOverArea[hit.tri] * (rayTmax * rayTmax) / cosLight;
        emissionWeight = powerHeuristic(payload.Pdf, pdfLight);
    }

    /* decals (Q9) */
    if (payload.DirectLightPdf != -1.0f && rayTmax > payload.DirectLightPdf)
        material.Color = mix(material.Color, payload.LightDirection, payload.LightDistance);

    payload.MaxRoughness = max(material.Roughness, payload.MaxRoughness);
    material.Roughness = max(payload.MaxRoughness, 0.01f);

    const mat3 geometryTBN = M3(vertex.Tangent, vertex.Bitangent, vertex.Normal);
    const vec3 N = normalize(vertex.Normal + geometryTBN * material.Normal);
    const mat3 TBN = computeTangentSpace(N);
    const mat3 invTBN = inverse(TBN);
    const vec3 V = normalize(invTBN * normalize(-rayDirWorld));

    uint32_t rngState = payload.RngState;

    BSDFSample bsdf = sampleBSDF(material, V, rngState);

    if (isHitFromInside)
    {
        bsdf.Color.x *= std::pow(material.AttenuationColor.x, rayTmax / material.AttenuationDistance);
        bsdf.Color.y *= std::pow(material.AttenuationColor.y, rayTmax / material.AttenuationDistance);
        bsdf.Color.z *= std::pow(material.AttenuationColor.z, rayTmax / material.AttenuationDistance);
    }

    const bool isRefracted = bsdf.Direction.z < 0.0f;

    const vec3 rayOrigin = offsetRayOriginShadowTerminator(vertex, v0, v1, v2, barycentricCoords, isRefracted);

    float lightPdf, lightSmplPdf;
    const float l0 = rnd(rngState);
    const float l1 = rnd(rngState);
    const float l2 = rnd(rngState);
    LightSample light = sampleLight(s, V3(l0, l1, l2), rayOrigin, lightPdf);
    emitterSample = 0;
    if (emissiveMode(em))
    {
        /* branch, alias draw and point from a secondary stream; the main stream is not advanced */
        uint32_t rng2 = jenkinsHash(rngState ^ 0x68bc21ebu);
        if (rnd(rng2) < em.pEmitter)
        {
            const uint32_t hi = xorshift(rng2), lo = xorshift(rng2);
            const uint32_t bucket = (uint32_t)(((uint64_t)hi * em.emitterIds.size()) >> 32);
            const uint32_t k = lo < em.aliasThreshold[bucket] ? bucket : em.aliasIndex[bucket];
            const float r1 = rnd(rng2);
            const float r2 = rnd(rng2);
            light = sampleEmitter(s, em, k, r1, r2, rayOrigin, lightPdf);
            emitterSample = 1;
            /* the last bounce: the reference mode never collects emission one vertex further, so neither does this */
            if (bounce + 1 >= p.bounce_count)
                lightPdf = 0.0f;
        }
        else
            lightPdf = lightPdf * (1.0f - em.pEmitter);
    }
    const vec3 L = normalize(invTBN * -light.Direction);
    const vec3 lightBsdf = evaluateBSDF(material, V, L, lightSmplPdf);
    if (emitterSample)
        light.Attenuation = powerHeuristic(lightPdf, lightSmplPdf);

    payload.Direction = normalize(TBN * bsdf.Direction);
    if (isRefracted)
        payload.Position = offsetRayOriginSelfIntersection(vertex.Position, -geometricNormal);
    else
        payload.Position = rayOrigin;
    payload.Bsdf = bsdf.Color;
    payload.Pdf = bsdf.Pdf;
    payload.Emissive = emissiveMode(em) ? material.EmissiveColor * emissionWeight : material.EmissiveColor;
    payload.RngState = rngState;
    payload.DirectLight = light.Color * light.Attenuation * lightBsdf;
    payload.DirectLightPdf = lightPdf;
    payload.LightDirection = light.Direction;
    payload.LightDistance = light.Distance;

    if (isRefracted)
        computeRefractedDifferentialRays(derivatives, vertex.Normal, rayOrigin, -viewDir, payload.Direction, dndu, dndv,
                                         material.Eta, rxOrigin, rxDirection, ryOrigin, ryDirection);
    else
        computeReflectedDifferentialRays(derivatives, vertex.Normal, rayOrigin, -viewDir, payload.Direction, dndu, dndv,
                                         rxOrigin, rxDirection, ryOrigin, ryDirection);

    payload.RayDifferentials0 = V4(rxOrigin, rxDirection.x);
    payload.RayDifferentials1 = V4(rxDirection.y, rxDirection.z, ryOrigin.x, ryOrigin.y);
    payload.RayDifferentials2 = V4(ryOrigin.z, ryDirection.x, ryDirection.y, ryDirection.z);
}

/* tracePrimaryType (raygen.rgen:68) with closestHitEmissive */
void tracePrimaryEmissive(const pto_scene &s, const EmitterTable &em, const pt_render_params &p, const Ray &ray,
                          Payload &payload, uint32_t bounce, uint32_t &emitterSample, Counters &c)
{
    emitterSample = 0;
    const HitInfo hit = traceClosest(s, ray.Origin, ray.Direction, ray.tmin, ray.tmax, c);
    /* the any-hit stage wrote its decal record into the payload before closest-hit / miss run */
    if (hit.decalDist != -1.0f)
    {
        payload.LightDirection = hit.decalColor;
        payload.LightDistance = hit.decalAlpha;
        payload.DirectLightPdf = hit.decalDist;
    }
    if (hit.tri == PT_NO_HIT)
        missShader(s, p, ray.Direction, payload);
    else
        closestHitEmissive(s, em, p, hit, ray.Origin, ray.Direction, payload, bounce, emitterSample, c);
}

/* raygenPixel (PT/Shaders/raygen.rgen:36-118) with tracePrimaryEmissive; a non-finite emitter sample is dropped */
vec3 raygenPixelEmissive(const pto_scene &s, const EmitterTable &em, const pt_render_params &p, uint32_t px, uint32_t py, uint32_t width, uint32_t height,
                 uint32_t sampleCount, uint32_t totalSamples, Counters &c)
{
    const mat4 ViewInverse = toMat4(p.view_inverse);
    const mat4 ProjInverse = toMat4(p.proj_inverse);
    uint32_t rngState = initRng(px, py, width, totalSamples);
    vec3 radiance = V3(0.0f);
    Payload payload;
    std::memset(&payload, 0, sizeof(payload));
    uint32_t restarts = 0;

    for (int smpl = 0; smpl < (int)sampleCount; smpl++)
    {
        vec3 throughput = V3(1.0f);
        const float ux = rnd(rngState);
        const float uy = rnd(rngState);
        vec2 u = V2(ux, uy);
        Ray ray, rx, ry;
        const vec2 pixel = V2((float)px, (float)py), resolution = V2((float)width, (float)height);
        if (p.lens_radius > 0)
        {
            const float u2x = rnd(rngState);
            const float u2y = rnd(rngState);
            ray = constructPrimaryRayLens(pixel, resolution, ViewInverse, ProjInverse, u, V2(u2x, u2y), p.lens_radius,
                                          p.focal_distance, rx, ry);
        }
        else
            ray = constructPrimaryRay(pixel, resolution, ViewInverse, ProjInverse, u, rx, ry);

        payload.RayDifferentials0 = V4(rx.Origin, rx.Direction.x);
        payload.RayDifferentials1 = V4(rx.Direction.y, rx.Direction.z, ry.Origin.x, ry.Origin.y);
        payload.RayDifferentials2 = V4(ry.Origin.z, ry.Direction.x, ry.Direction.y, ry.Direction.z);
        payload.MaxRoughness = 0.0f;

        for (uint32_t bounce = 0; bounce < p.bounce_count; bounce++)
        {
            payload.RngState = rngState;
            payload.DirectLightPdf = -1.0f;
            payload.LightDirection = V3(0.0f);
            payload.LightDistance = 0.0f;
            uint32_t emitterSample;
            tracePrimaryEmissive(s, em, p, ray, payload, bounce, emitterSample, c);
            rngState = payload.RngState;

            if (payload.Pdf == -1.0f)
            {
                radiance += throughput * payload.Emissive;
                break;
            }
            radiance += throughput * payload.Emissive;

            if (payload.DirectLightPdf > 0.0f)
            {
                const vec3 contribution = throughput * payload.DirectLight / payload.DirectLightPdf;
                const bool dropped = emitterSample && !(std::isfinite(contribution.x) && std::isfinite(contribution.y) &&
                                                                std::isfinite(contribution.z));
                if (!dropped && !checkOccluded(s, payload.LightDirection, payload.Position, payload.LightDistance, c))
                    radiance += contribution;
            }

            if (payload.Pdf > 0.001f)
                throughput *= payload.Bsdf / payload.Pdf;

            const float prob = min(maxComponent(throughput), 1.0f);
            if (prob < 0.001f)
                break;
            if (prob < rnd(rngState))
                break;
            throughput /= prob;

            ray.Origin = payload.Position;
            ray.Direction = payload.Direction;
        }
        c.samples++;

        if (isnan(radiance.x) || isnan(radiance.y) || isnan(radiance.z) || isinf(radiance.x) || isinf(radiance.y) ||
            isinf(radiance.z))
        {
            radiance = V3(0.0f);
            if (++restarts > kMaxRestarts)
                break;
            c.restarts++;
            smpl = -1;
            continue;
        }
    }
    return radiance;
}

} // namespace

struct ptx_emitters : EmitterTable
{
};

extern "C" {

/* the emitter table of a scene (built from the scene's current sampler state) */
PT_API ptx_emitters *ptx_emitters_create(const pto_scene *s)
{
    if (!s)
        return nullptr;
    ptx_emitters *t = new ptx_emitters();
    buildEmitterTable(*s, *t);
    return t;
}

PT_API void ptx_emitters_destroy(ptx_emitters *t) { delete t; }

PT_API int32_t ptx_emitter_table(const ptx_emitters *t, uint32_t *out_count, uint32_t *flat_ids, uint32_t *weights,
                                 uint32_t *alias_threshold, uint32_t *alias_index, uint32_t capacity)
{
    if (!t || !out_count)
        return PT_ERR_INVALID_ARGUMENT;
    const uint32_t n = (uint32_t)t->emitterIds.size();
    *out_count = n;
    if ((flat_ids || weights || alias_threshold || alias_index) && capacity < n)
        return PT_ERR_INVALID_ARGUMENT;
    for (uint32_t k = 0; k < n; k++)
    {
        if (flat_ids)
            flat_ids[k] = t->emitterIds[k];
        if (weights)
            weights[k] = t->emitterWeights[k];
        if (alias_threshold)
            alias_threshold[k] = t->aliasThreshold[k];
        if (alias_index)
            alias_index[k] = t->aliasIndex[k];
    }
    return PT_OK;
}

/* pto_render_frames in the emissive-MIS mode */
PT_API int32_t ptx_render_frames(const pto_scene *s, const ptx_emitters *em, const pt_render_params *p, uint32_t width,
                                 uint32_t height, uint32_t first_sample, uint32_t frame_count, uint32_t samples_per_frame,
                                 const pt_tile *tiles, uint32_t tile_count, float *accum, int32_t threads, pto_counters *out)
{
    if (!s || !em || !p || !accum || samples_per_frame == 0)
        return PT_ERR_INVALID_ARGUMENT;
    int nthreads = threads > 0 ? threads : (int)std::thread::hardware_concurrency();
    if (nthreads < 1)
        nthreads = 1;
    std::vector<Counters> counters(nthreads);
    std::atomic<uint32_t> nextRow { 0 };
    auto worker = [&](int tid) {
        Counters &c = counters[tid];
        for (;;)
        {
            const uint32_t y = nextRow.fetch_add(1);
            if (y >= height)
                break;
            for (uint32_t x = 0; x < width; x++)
            {
                if (!inTiles(x, y, tiles, tile_count))
                    continue;
                float *px = accum + ((size_t)y * width + x) * 4;
                for (uint32_t f = 0; f < frame_count; f++)
                {
                    const vec3 radiance = raygenPixelEmissive(*s, *em, *p, x, y, width, height, samples_per_frame,
                                                              first_sample + f * samples_per_frame, c);
                    px[0] = radiance.x + px[0];
                    px[1] = radiance.y + px[1];
                    px[2] = radiance.z + px[2];
                    px[3] = 1.0f;
                }
            }
        }
    };
    if (nthreads == 1)
        worker(0);
    else
    {
        std::vector<std::thread> pool;
        for (int i = 0; i < nthreads; i++)
            pool.emplace_back(worker, i);
        for (auto &t : pool)
            t.join();
    }
    if (out)
    {
        Counters total;
        for (auto &c : counters)
            total.add(c);
        out->rays_closest = total.rays_closest;
        out->rays_shadow = total.rays_shadow;
        out->samples = total.samples;
        out->hits = total.hits;
        out->box_tests_closest = total.box_c;
        out->tri_tests_closest = total.tri_c;
        out->box_tests_shadow = total.box_s;
        out->tri_tests_shadow = total.tri_s;
        out->alpha_tests_closest = total.alpha_c;
        out->alpha_tests_shadow = total.alpha_s;
        out->texel_fetches = total.texels;
        out->restarts = total.restarts;
    }
    return PT_OK;
}

} // extern "C"
