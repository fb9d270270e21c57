/*
 * pt_core.h — C ABI of the B200-native path-tracing core.
 *
 * This is the drop-in boundary for the hot path of piotrprzybyszdev/Path-Tracing:
 * the work the reference does in Renderer::UpdateSceneData + Renderer::Render
 * (vkCmdTraceRaysKHR over raygen.rgen / closestHit.rchit / anyhit.rahit /
 * occlusionAnyhit.rahit / miss.rmiss / occlusion.rmiss with a driver-built
 * TLAS/BLAS).  The reference has no FFI for this path (Renderer is a static
 * C++ class, Path-Tracing/Renderer/Renderer.h:42-85); every entry point below
 * cites the reference interface it replaces.  All citations are relative to
 * the reference checkout (Path-Tracing/ = PT/).
 *
 * Conventions
 *   - plain C, no torch / CUDA types in any signature; pointers are HOST
 *     pointers unless the name says "device";
 *   - every function returns pt_status (0 = ok, negative = error); the text of
 *     the last error is available through pt_last_error();
 *   - caller owns all host arrays; nothing is retained after a call returns;
 *   - a pt_context is externally synchronised (one thread at a time), like the
 *     reference's Renderer, which is only ever called from the main thread;
 *   - there is NO CPU fallback: without a CUDA device pt_context_create fails.
 */
#ifndef PT_CORE_H
#define PT_CORE_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(_WIN32)
#define PT_API __declspec(dllexport)
#else
#define PT_API __attribute__((visibility("default")))
#endif

/* ------------------------------------------------------------------------- */
/* status                                                                    */
/* ------------------------------------------------------------------------- */

typedef int32_t pt_status;
enum {
    PT_OK = 0,
    PT_ERR_INVALID_ARGUMENT = -1, /* null pointer, index out of range, bad enum                */
    PT_ERR_NO_DEVICE = -2,        /* no CUDA device / wrong architecture (no CPU fallback)       */
    PT_ERR_CUDA = -3,             /* a CUDA call failed; see pt_last_error                       */
    PT_ERR_OUT_OF_MEMORY = -4,
    PT_ERR_NO_SCENE = -5,         /* render/trace before pt_scene_upload                         */
    PT_ERR_NO_TARGET = -6,        /* render/readback before pt_render_begin                      */
    PT_ERR_UNSUPPORTED = -7       /* e.g. animated geometry, BC textures (SURVEY §8f)            */
};

typedef struct pt_context pt_context;

/* ------------------------------------------------------------------------- */
/* scene data contract — byte-identical to the reference's host structs      */
/* ------------------------------------------------------------------------- */

/* Shaders::Vertex, PT/Shaders/ShaderTypes.incl:40-47 (56 bytes, scalar-aligned). */
typedef struct pt_vertex {
    float position[3];
    float texcoords[2];
    float normal[3];
    float tangent[3];
    float bitangent[3];
} pt_vertex;

/* Shaders::AnimatedVertex, PT/Shaders/ShaderTypes.incl:50-59 (88 bytes): a Vertex + 4 bone indices
 * and weights (MaxBonesPerVertex = 4, ShaderTypes.incl:31). */
typedef struct pt_animated_vertex {
    float position[3];
    float texcoords[2];
    float normal[3];
    float tangent[3];
    float bitangent[3];
    uint32_t bone_indices[4];
    float bone_weights[4];
} pt_animated_vertex;

/* PathTracing::Geometry, PT/Scene.h:63-71 (bools widened to u32; IsAnimated travels separately in
 * pt_scene_desc::geometry_is_animated so that this struct keeps its 20 bytes). */
typedef struct pt_geometry {
    uint32_t vertex_offset; /* first vertex; indices are relative to it (PT/Shaders/common.glsl:27-34) */
    uint32_t vertex_length;
    uint32_t index_offset;
    uint32_t index_length;
    uint32_t is_opaque; /* 0 => alpha-tested any-hit runs (PT/Renderer/AccelerationStructure.cpp:94-97) */
} pt_geometry;

/* Shaders::SBTBuffer, PT/Shaders/ShaderRendererTypes.incl:42-47; one per (model, mesh) in model
 * order, exactly the records Renderer::UpdateSceneData adds (PT/Renderer/Renderer.cpp:381-399). */
typedef struct pt_mesh_record {
    uint32_t geometry_index;
    uint32_t material_id;     /* (index << 8) | type, PT/Shaders/ShaderTypes.incl:155-168 */
    uint32_t transform_index; /* into transforms[]; 0 = identity (PT/Scene.h:306)          */
} pt_mesh_record;

/* PathTracing::Model, PT/Scene.h:96-100. */
typedef struct pt_model {
    uint32_t mesh_offset; /* index of the model's first pt_mesh_record */
    uint32_t mesh_count;
} pt_model;

/* PathTracing::ModelInstance, PT/Scene.h:102-107, in the form BuildTlas hands to Vulkan
 * (PT/Renderer/AccelerationStructure.cpp:268-275): first 12 floats of the row-vector
 * glm::mat4 == a 3x4 row-major object-to-world matrix. */
typedef struct pt_instance {
    float transform[12];
    uint32_t model_index;
} pt_instance;

enum {
    PT_MATERIAL_METALLIC_ROUGHNESS = 0, /* PT/Shaders/ShaderTypes.incl:143-145 */
    PT_MATERIAL_SPECULAR_GLOSSINESS = 1,
    PT_MATERIAL_PHONG = 2
};

/* Shaders::MetallicRoughnessMaterial, PT/Shaders/ShaderTypes.incl:61-80 (96 bytes). */
typedef struct pt_material_mr {
    float emissive_color[3];
    float emissive_intensity;
    float color[4];
    float roughness;
    float metalness;
    float ior;
    float transmission;
    float attenuation_color[3];
    float attenuation_distance;
    float pad0, pad1, pad2;
    uint32_t emissive_idx;
    uint32_t color_idx;
    uint32_t normal_idx;
    uint32_t roughness_idx;
    uint32_t metallic_idx;
} pt_material_mr;

/* Shaders::SpecularGlossinessMaterial, PT/Shaders/ShaderTypes.incl:82-99 (96 bytes).
 * Shaders::PhongMaterial (:101-118) has the same layout with Shininess for Glossiness. */
typedef struct pt_material_sg {
    float emissive_color[3];
    float emissive_intensity;
    float color[4];
    float specular[3];
    float glossiness; /* Phong: shininess */
    float attenuation_color[3];
    float attenuation_distance;
    float ior;
    float transmission;
    uint32_t emissive_idx;
    uint32_t color_idx;
    uint32_t normal_idx;
    uint32_t specular_idx;
    uint32_t glossiness_idx; /* Phong: shininess_idx */
    float pad0;
} pt_material_sg;

typedef pt_material_sg pt_material_phong;

/* Shaders::DirectionalLight / PointLight, PT/Shaders/ShaderTypes.incl:120-141. */
typedef struct pt_directional_light {
    float color[3];
    float pad0;
    float direction[3];
    float pad1;
} pt_directional_light;

typedef struct pt_point_light {
    float color[3];
    float pad0;
    float position[3];
    float pad1;
    float attenuation_constant;
    float attenuation_linear;
    float attenuation_quadratic;
    float pad2;
} pt_point_light;

#define PT_MAX_LIGHT_COUNT 64u       /* PT/Shaders/ShaderTypes.incl:30 */
#define PT_SCENE_TEXTURE_OFFSET 9u   /* PT/Shaders/ShaderTypes.incl:27; slots 0-8 are built in */

enum {
    PT_TEXTURE_RGBA8 = 0,   /* TextureFormat::RGBAU8,  PT/Scene.h:35-42 */
    PT_TEXTURE_RGBAF32 = 1, /* TextureFormat::RGBAF32 */
    PT_TEXTURE_BC1 = 2,     /* TextureFormat::BC1: DXT1 blocks (8 B per 4x4), 1-bit alpha          */
    PT_TEXTURE_BC3 = 3,     /* TextureFormat::BC3: DXT5 blocks (16 B), always sampled as sRGB       */
    PT_TEXTURE_BC5 = 4      /* TextureFormat::BC5: ATI2N blocks (16 B), two channels, sampled (r, g, 0, 1) */
};

/* One decoded level-0 image (what TextureImporter::LoadTextureData returns,
 * PT/TextureImporter.cpp:413-424).  The core builds the full mip chain itself
 * (PT/Renderer/Image.cpp:14-17,264-305); block-compressed images (SURVEY §8f rank 4) are decoded to
 * RGBA8 on the GPU at upload, level by level.  srgb follows the reference's rule
 * Color/Specular/Emissive/Skybox => sRGB (PT/Renderer/TextureUploader.cpp:571-595). */
typedef struct pt_texture_desc {
    uint32_t width;
    uint32_t height;
    uint32_t format; /* PT_TEXTURE_* */
    uint32_t srgb;   /* RGBA8 and BC1 (BC3 is always sRGB, BC5 and float never: TextureUploader.cpp:571-595) */
    const void *pixels;
    /* Block-compressed formats only: number of mip levels stored in `pixels`, level 0 first, tightly
     * packed, exactly as TextureImporter's gli loader concatenates a .dds file
     * (PT/TextureImporter.cpp:311-343).  Mips of compressed textures are never generated
     * (TextureUploader.cpp:420-456): the sampler clamps to the last stored level.  0 means 1. */
    uint32_t levels;
} pt_texture_desc;

enum {
    PT_MISS_FLAGS_NONE = 0x0,      /* PT/Shaders/ShaderRendererTypes.incl:92-95 */
    PT_MISS_FLAGS_SKYBOX_2D = 0x1,
    PT_MISS_FLAGS_SKYBOX_CUBE = 0x2
};
enum {
    PT_HIT_FLAGS_NONE = 0x0,       /* PT/Shaders/ShaderRendererTypes.incl:97-99 */
    PT_HIT_FLAGS_DX_NORMAL_TEXTURES = 0x1
};

/* Everything Renderer::UpdateSceneData pulls out of a Scene (PT/Scene.h:182-212;
 * use sites PT/Renderer/Renderer.cpp:257-331, 381-399, 1719-1726). */
typedef struct pt_scene_desc {
    const pt_vertex *vertices;
    uint64_t vertex_count;
    const uint32_t *indices;
    uint64_t index_count;
    const float *transforms; /* transform_count x 12 floats, 3x4 row-major; [0] = identity */
    uint32_t transform_count;
    const pt_geometry *geometries;
    uint32_t geometry_count;
    const pt_mesh_record *mesh_records;
    uint32_t mesh_record_count;
    const pt_model *models;
    uint32_t model_count;
    const pt_instance *instances;
    uint32_t instance_count;
    const pt_material_mr *mr_materials;
    uint32_t mr_material_count;
    const pt_material_sg *sg_materials;
    uint32_t sg_material_count;
    const pt_material_phong *phong_materials;
    uint32_t phong_material_count;
    const pt_texture_desc *textures; /* scene texture i lives in slot PT_SCENE_TEXTURE_OFFSET + i */
    uint32_t texture_count;
    const pt_point_light *point_lights;
    uint32_t point_light_count; /* <= PT_MAX_LIGHT_COUNT */
    pt_directional_light directional_light;
    const pt_texture_desc *skybox_2d; /* equirect sky for PT_MISS_FLAGS_SKYBOX_2D, or NULL */
    /* Six equally sized faces for PT_MISS_FLAGS_SKYBOX_CUBE, or NULL, in the order
     * TextureUploader::UploadSkyboxBlocking fills the cube image's layers
     * (PT/Renderer/TextureUploader.cpp:232-236): Front, Back, Up, Down, Left, Right
     * = Vulkan cube faces +X, -X, +Y, -Y, +Z, -Z. */
    const pt_texture_desc *skybox_cube;
    /* Skeletal animation (SURVEY §8f rank 3; Scene::GetAnimatedVertices / GetAnimatedIndices /
     * GetBoneTransforms, PT/Scene.h:183-196).  geometry_is_animated[i] != 0 marks geometry i as
     * Geometry::IsAnimated: its vertex_offset / index_offset then address animated_vertices /
     * animated_indices instead of vertices / indices (PT/Renderer/Renderer.cpp:286-372).  The core
     * skins them with bone_transforms (skinning.comp:21-50) before it bakes and builds.  All NULL / 0
     * for a scene without skeletal animation. */
    const uint32_t *geometry_is_animated; /* geometry_count entries, or NULL */
    const pt_animated_vertex *animated_vertices;
    uint64_t animated_vertex_count;
    const uint32_t *animated_indices;
    uint64_t animated_index_count;
    const float *bone_transforms; /* bone_count x 12 floats: glm::mat3x4 = three vec4 columns = the rows of
                                     the 3x4 bone matrix (Bone::Offset * node transform, Scene.cpp:72-73) */
    uint32_t bone_count;
} pt_scene_desc;

/* Shaders::RaygenUniformData (PT/Shaders/ShaderRendererTypes.incl:26-34) plus the two
 * specialisation constants (:89-99).  SampleCount/TotalSamples are arguments of
 * pt_render_samples.  Matrices are column-major exactly as glm stores them. */
typedef struct pt_render_params {
    float view_inverse[16];
    float proj_inverse[16];
    uint32_t bounce_count;
    float lens_radius;
    float focal_distance;
    uint32_t miss_flags;
    uint32_t hit_flags;
} pt_render_params;

/* Pixel rectangle [x0,x1) x [y0,y1) of the full image; used to partition one frame over GPUs. */
typedef struct pt_tile {
    uint32_t x0, y0, x1, y1;
} pt_tile;

/* A ray query and its result (traceRayEXT contract, PT/Shaders/raygen.rgen:31,68). */
typedef struct pt_ray {
    float origin[3];
    float tmin;
    float direction[3];
    float tmax;
} pt_ray;

#define PT_NO_HIT 0xffffffffu

typedef struct pt_hit {
    uint32_t instance;   /* gl_InstanceID; PT_NO_HIT on a miss                         */
    uint32_t geometry;   /* geometry index inside the model's BLAS (gl_GeometryIndexEXT) */
    uint32_t primitive;  /* gl_PrimitiveID                                              */
    float t;             /* gl_RayTmaxEXT at the closest hit                            */
    float u, v;          /* hitAttributeEXT barycentrics (weights of v1, v2)            */
} pt_hit;

/* Kernel classes of the wavefront (indices of pt_stats.kernel_ms / kernel_launch_count). */
enum {
    PT_KERNEL_EXTEND = 0, /* closest-hit traversal                        */
    PT_KERNEL_SHADE = 1,  /* miss / closest-hit shading + bounce logic     */
    PT_KERNEL_SHADOW = 2, /* occlusion traversal                           */
    PT_KERNEL_FINISH = 3, /* accumulate / restart / regenerate + compaction */
    PT_KERNEL_CLASS_COUNT = 4
};

/* Device counters of the last pt_render_samples call plus build info. */
typedef struct pt_stats {
    uint64_t rays_closest;        /* closest-hit queries traced (raygen.rgen:68)                 */
    uint64_t rays_shadow;         /* occlusion queries traced (raygen.rgen:31)                    */
    uint64_t samples;             /* finished iterations of the sample loop (raygen.rgen:42)      */
    uint64_t hits;                /* closest-hit queries that hit                                 */
    uint64_t box_tests_closest;   /* child AABBs tested by closest-hit rays   (traversal stats)   */
    uint64_t tri_tests_closest;   /* ray-triangle tests of closest-hit rays   (traversal stats)   */
    uint64_t alpha_tests_closest; /* anyhit.rahit evaluations                 (traversal stats)   */
    uint64_t box_tests_shadow;    /*                                          (traversal stats)   */
    uint64_t tri_tests_shadow;    /*                                          (traversal stats)   */
    uint64_t alpha_tests_shadow;  /* occlusionAnyhit.rahit evaluations        (traversal stats)   */
    uint64_t texel_fetches;       /* texels read by the material fetches      (traversal stats)   */
    uint64_t restarts;            /* NaN/Inf sample restarts (raygen.rgen:99-112)                 */
    uint64_t wavefront_iterations;
    uint64_t kernel_launches;     /* launches of this library's kernels in the last render call   */
    uint64_t triangle_count;      /* flattened (instanced) triangles in the BVH                   */
    uint64_t bvh_node_count;
    uint64_t bvh_bytes;
    float bvh_build_ms;
    float scene_upload_ms;
    float last_render_ms;         /* CUDA-event time of the last pt_render_samples                */
    float kernel_ms[PT_KERNEL_CLASS_COUNT];              /* with pt_set_kernel_timing(1) only     */
    uint32_t kernel_launch_count[PT_KERNEL_CLASS_COUNT];
    /* traversal-tail diagnostics (traversal stats only): rays by the number of BVH nodes they visited,
     * bins [0,16) [16,32) [32,64) [64,128) [128,256) [256,512) [512,1024) [1024,inf); and the
     * warp-level loop iterations of the traversal kernels, in total and in drain mode (queue empty) */
    uint64_t node_visit_hist[8];
    uint64_t warp_iterations;
    uint64_t warp_drain_iterations;
    uint64_t max_warp_drain_iterations;
    uint64_t bvh_reference_count; /* leaf entries of the BVH: >= triangle_count (a large diagonal triangle enters the BVH
                                     as several references to the same triangle, bvh_build.cu k_split_*)            */
    uint32_t bvh_max_depth;   /* levels of the wide BVH of the uploaded scene                                     */
    uint32_t stack_overflows; /* entries the traversal stack could not hold in the last call: non-zero FAILS the
                                 call (PT_ERR_UNSUPPORTED) — a dropped entry is a skipped sub-tree              */
} pt_stats;

/* ------------------------------------------------------------------------- */
/* context                                                                   */
/* ------------------------------------------------------------------------- */

/* Replaces DeviceContext::Init + Renderer::Init (PT/Renderer/DeviceContext.cpp:30,
 * PT/Renderer/Renderer.cpp:77): binds the CUDA device's primary context, creates the
 * stream and the nine built-in 1x1 textures (Renderer.cpp:127-173). */
PT_API pt_status pt_context_create(int32_t cuda_device, pt_context **out_ctx);

/* Replaces Renderer::Shutdown (PT/Renderer/Renderer.cpp:176-218). */
PT_API void pt_context_destroy(pt_context *ctx);

/* Error text of the last failed call on ctx (ctx may be NULL for create failures).
 * Replaces the PathTracing::error exception text (PT/Core/Core.cpp:82-90). */
PT_API const char *pt_last_error(const pt_context *ctx);

/* ------------------------------------------------------------------------- */
/* scene                                                                     */
/* ------------------------------------------------------------------------- */

/* Replaces Renderer::UpdateSceneData for a new scene (PT/Renderer/Renderer.cpp:238-439)
 * and the AccelerationStructure constructor (PT/Renderer/AccelerationStructure.cpp:12-35):
 * copies the scene to the device, bakes instance x mesh transforms, builds the BVH on
 * the GPU, builds texture mip chains.  Blocking. */
PT_API pt_status pt_scene_upload(pt_context *ctx, const pt_scene_desc *scene);

/* What Scene::Update changes from frame to frame in an animated scene (PT/Scene.cpp:52-83).
 * A NULL pointer leaves that part of the scene as it is. */
typedef struct pt_scene_update_desc {
    const float *instance_transforms; /* instance_count x 12 floats, the pt_instance::transform of every
                                         instance in upload order (ModelInstance::Transform, Scene.cpp:69-70) */
    uint32_t instance_count;          /* must equal the uploaded scene's instance_count */
    const pt_point_light *point_lights; /* the whole light array (positions follow their nodes, Scene.cpp:75-77) */
    uint32_t point_light_count;       /* <= PT_MAX_LIGHT_COUNT */
    const pt_directional_light *directional_light; /* Scene.cpp:79-80 */
    const float *bone_transforms;     /* bone_count x 12 floats (Scene::GetBoneTransforms, Scene.cpp:72-73):
                                         re-skins the animated geometries (RecordSkinningCommands) */
    uint32_t bone_count;              /* must equal the uploaded scene's bone_count */
} pt_scene_update_desc;

/* Replaces the per-frame half of Renderer::UpdateSceneData / Renderer::Render for animated scenes:
 * the light uniform rewrite (PT/Renderer/Renderer.cpp:1719-1726) and
 * AccelerationStructure::RecordUpdateCommands (PT/Renderer/AccelerationStructure.cpp:48-57, called
 * from Renderer.cpp:1753-1754).  Where the reference refits BLAS + TLAS, the core re-bakes the
 * instances and rebuilds its BVH on the GPU; new bone transforms first re-skin the animated
 * geometries (Renderer::RecordSkinningCommands, Renderer.cpp:854-890 = skinning.comp).  Static
 * geometry, materials and textures are unchanged.
 * The accumulation buffer is NOT reset — the caller does that (Renderer::UpdateSceneData's
 * `updated` flag, Renderer.cpp:240-241) with pt_render_begin.  Blocking. */
PT_API pt_status pt_scene_update(pt_context *ctx, const pt_scene_update_desc *desc);

/* Replaces the sampler state of Renderer::CreateSampler (PT/Renderer/Renderer.cpp:103-112: linear mag / min / mip,
 * repeat, anisotropyEnable with maxAnisotropy = the device limit): the maximum anisotropy of the material fetches
 * (textureGrad, material.glsl:62-171).  1 = isotropic trilinear filtering (GL 4.6 8.14); up to 16 taps along the major
 * axis of the footprint otherwise (the example implementation of the Vulkan specification, "Texel Anisotropic
 * Filtering"; a footprint that reaches the 1 x 1 top level is one tap).  16 = what the reference's sampler asks for on
 * every current GPU.  DEFAULT 1: without texture units every tap is eight software texel fetches, and path tracing's
 * secondary bounces have huge, elongated footprints — the 16-tap sampler makes k_shade 4-7 x slower (measured, DESIGN.md)
 * for a filter whose exact result is implementation-defined in the reference anyway.  Takes effect at the next render
 * call; the accumulated image is not reset. */
PT_API pt_status pt_set_sampler(pt_context *ctx, uint32_t max_anisotropy);

/* Light sampling of next-event estimation (an extension: the reference has no counterpart).
 *   PT_LIGHT_SAMPLING_REFERENCE     the reference's: one analytic light (point or directional) per hit (default).
 *   PT_LIGHT_SAMPLING_EMISSIVE_MIS  also samples the scene's emissive triangles (opaque geometry whose material has
 *                                   emissive_intensity > 0 and a non-black emissive colour or texture), in proportion to
 *                                   area x luminance, and weights emission found by BSDF sampling with the power
 *                                   heuristic.  Every path vertex, and with it rays_closest / hits, is that of the
 *                                   reference mode; only the collected radiance differs.  A scene without emitters
 *                                   renders bit for bit as in the reference mode.  Semantics: DESIGN.md section 3g.
 * Takes effect at the next render call; the accumulated image is not reset. */
typedef enum pt_light_sampling {
    PT_LIGHT_SAMPLING_REFERENCE = 0,
    PT_LIGHT_SAMPLING_EMISSIVE_MIS = 1,
} pt_light_sampling;
PT_API pt_status pt_set_light_sampling(pt_context *ctx, uint32_t mode);

/* The emitter table of PT_LIGHT_SAMPLING_EMISSIVE_MIS (built now if it is out of date): *out_count emitters; entry k is
 * flat triangle flat_ids[k] (flattening order: instance, mesh in model, primitive) with integer weight weights[k], drawn
 * through the alias entry (alias_threshold[k], alias_index[k]): a uniform bucket k and a uniform 32-bit fraction x keep k
 * when x < alias_threshold[k], else take alias_index[k].  Arrays may be NULL (count only); otherwise they hold capacity
 * entries, and PT_ERR_INVALID_ARGUMENT is returned when capacity < count. */
PT_API pt_status pt_emitter_table(pt_context *ctx, uint32_t *out_count, uint32_t *flat_ids, uint32_t *weights,
                                  uint32_t *alias_threshold, uint32_t *alias_index, uint32_t capacity);

/* Replaces Renderer::UpdateTexture(index) (PT/Renderer/Renderer.cpp:441-471): replace the
 * content of one texture slot (slot = PT_SCENE_TEXTURE_OFFSET + scene texture index). */
PT_API pt_status pt_texture_upload(pt_context *ctx, uint32_t slot, const pt_texture_desc *texture);

/* ------------------------------------------------------------------------- */
/* rendering                                                                 */
/* ------------------------------------------------------------------------- */

/* Replaces the accumulation-image (re)creation and clear (PT/Renderer/Renderer.cpp:1284-1288,
 * 1734-1748, OnResize / SetSettings(RenderSettings) :825-852): allocates a zeroed
 * width x height float4 sum buffer and the wavefront path state. */
PT_API pt_status pt_render_begin(pt_context *ctx, uint32_t width, uint32_t height);

/* Replaces Renderer::Render's trace pass (PT/Renderer/Renderer.cpp:1686-1700, 892-917)
 * run sample_count times with SampleCount = 1 and TotalSamples = first_sample + i — the
 * schedule the reference's Profile/Debug builds use (PT/Core/Config.h:34-36).  tiles == NULL
 * renders the whole frame; otherwise only pixels inside the tile_count rectangles are
 * rendered (RNG still uses global pixel coordinates and the full resolution, so the result is
 * bit-identical to the same pixels of a full-frame render).  Blocking: returns when every
 * sample has been accumulated (the host polls the wavefront's active-path counter). */
PT_API pt_status pt_render_samples(pt_context *ctx, const pt_render_params *params, uint32_t first_sample,
                                   uint32_t sample_count, const pt_tile *tiles, uint32_t tile_count);

/* The same with the reference's Release-profile frame structure (Config::SamplesPerFrame > 1 and the adaptive
 * Renderer::s_SamplesPerFrame, PT/Renderer/Renderer.cpp:1631-1657, 1688-1700): frame f is one vkCmdTraceRaysKHR with
 * SampleCount = samples_per_frame and TotalSamples = first_sample + f * samples_per_frame, i.e. raygen.rgen:36-118 runs
 * the samples of a pixel on ONE rng stream (seeded from TotalSamples), sums their radiance before touching the image
 * and restarts ALL of them when the running sum turns NaN / Inf (raygen.rgen:99-112).  samples_per_frame = 1 is
 * pt_render_samples.  1 <= samples_per_frame <= 8192. */
PT_API pt_status pt_render_frames(pt_context *ctx, const pt_render_params *params, uint32_t first_sample,
                                  uint32_t frame_count, uint32_t samples_per_frame, const pt_tile *tiles,
                                  uint32_t tile_count);

/* Device address of the float4 accumulation (sum) buffer, row pitch in bytes, and the CUDA
 * stream (cudaStream_t as void*) work is queued on — for an NCCL reduce/gather in the caller. */
PT_API pt_status pt_accum_device_ptr(pt_context *ctx, void **out_float4_device_ptr, size_t *out_pitch_bytes,
                                     void **out_cuda_stream);

/* Replaces OutputSaver's GPU->host copy (PT/Renderer/OutputSaver.cpp:113-181) for the raw
 * float4 sum image: copies width*height*4 floats (RGB = sum of samples, A = 1) to host. */
PT_API pt_status pt_readback(pt_context *ctx, float *out_rgba, size_t out_bytes);

/* ---- post-processing and output conversion (SURVEY §8f rank 2) ---------- */

/* Renderer::PostProcessSettings (PT/Renderer/Renderer.h:68-73) + the tone-mapping
 * specialisation constant (PT/Shaders/ShaderRendererTypes.incl:70-72). */
typedef struct pt_postprocess_params {
    float exposure;        /* default 1.0 */
    float bloom_threshold; /* default 1.0 */
    float bloom_intensity; /* default 0.1 */
    uint32_t tone_mapping; /* PT_TONE_MAPPING_SDR: 1 - exp(-c); PT_TONE_MAPPING_HDR: identity */
} pt_postprocess_params;

enum { PT_TONE_MAPPING_SDR = 0, PT_TONE_MAPPING_HDR = 1 };

/* OutputSaver::SelectImageFormat (PT/Renderer/OutputSaver.cpp:255-273): png/jpg/tga/mp4 outputs
 * are R8G8B8A8_SRGB, hdr outputs R32G32B32A32_SFLOAT. */
enum { PT_OUTPUT_RGBA8_SRGB = 0, PT_OUTPUT_RGBAF32 = 1 };

/* Replaces Renderer::RecordPostProcessCommands + RecordSaveOutputCommands
 * (PT/Renderer/Renderer.cpp:928-1060, 1205-1250) and OutputSaver's blit + read-back
 * (PT/Renderer/OutputSaver.cpp:113-181) for the accumulated image:
 *   postprocess.comp:16-40   colour = sum / total_samples * exposure (NaN -> red, Inf -> green
 *                            markers), soft-knee bloom prefilter; both stored as RGBA16F
 *   bloomDownsample.comp / bloomUpsample.comp over mip levels 0 .. min(levels - 3, 12) - 1
 *                            of the RGBA16F bloom image (bilinear, clamp-to-edge sampler)
 *   composition.comp:15-25   colour += bloom_intensity * 0.1 * bloom
 *   toneMapping.comp:13-24   in place on the RGBA16F "linear output image"
 *   blit to the output format (sRGB encode + 8-bit quantisation, or float widening).
 * Writes width*height*4 bytes (RGBA8) or width*height*16 bytes (RGBAF32) to host memory;
 * alpha is 1.  The accumulation buffer is not modified. */
PT_API pt_status pt_postprocess(pt_context *ctx, const pt_postprocess_params *params, uint32_t total_samples,
                                uint32_t output_format, void *out_pixels, size_t out_bytes);

/* ---- denoiser (DESIGN §3h) ------------------------------------------------ */

/* Edge-avoiding a-trous wavelet filter (SVGF's spatial filter, Schied et al. 2017) guided by the
 * pixel-centre primary hit's base colour, shading normal and hit distance. */
typedef struct pt_denoise_params {
    uint32_t iterations;   /* a-trous levels K, 0..8 (step 2^k); 0 = the mean radiance, unchanged */
    float sigma_luminance; /* colour edge-stopping, in standard deviations (SVGF sigma_l; suggested 4)  */
    float sigma_normal;    /* exponent of the normal weight (suggested 128)                           */
    float sigma_depth;     /* depth edge-stopping (suggested 1)                                       */
} pt_denoise_params;

/* Denoises accumulation / total_samples of the current target. Writes width*height RGBA floats of mean radiance
 * (A = 1) to out_rgba if it is not NULL, and keeps the result on the device for pt_postprocess_denoised.
 * params supplies the camera the image was rendered with (the guides are traced with it); lens_radius > 0 is
 * PT_ERR_UNSUPPORTED (pinhole guides cannot describe a defocused image). The accumulation buffer is not modified. */
PT_API pt_status pt_denoise(pt_context *ctx, const pt_render_params *params, const pt_denoise_params *denoise,
                            uint32_t total_samples, float *out_rgba, size_t out_bytes);

/* The guide buffers of the last pt_denoise: per pixel (albedo.rgb, hit distance t; t = -1 on a miss) and
 * (shading normal.xyz, 0). For tests and for callers with their own denoiser. Either pointer may be NULL. */
PT_API pt_status pt_denoise_guides(pt_context *ctx, float *out_albedo_t, float *out_normal, size_t out_bytes);

/* pt_postprocess's chain (exposure, bloom, tone map, output format) on the last pt_denoise result. */
PT_API pt_status pt_postprocess_denoised(pt_context *ctx, const pt_postprocess_params *params, uint32_t output_format,
                                         void *out_pixels, size_t out_bytes);

/* ---- temporal denoiser (DESIGN §3j) --------------------------------------- */

/* SVGF's temporal stage (Schied et al. 2017, §4.1-4.2): the demodulated irradiance of each call is accumulated into a
 * per-pixel history reprojected from the previous call's camera, and the spatial filter runs on the result. */
typedef struct pt_temporal_params {
    float alpha;          /* weight of the new frame once the history is long: a = max(alpha, 1/n); 0..1 (SVGF: 0.2) */
    float alpha_moments;  /* the same for the luminance moments, 0..1 (SVGF: 0.2)                                 */
    uint32_t reset;       /* 1: discard the history before this frame                                              */
} pt_temporal_params;

/* One frame of temporal denoising: accumulation / total_samples of the current target is reprojected against the
 * history of the previous call, accumulated, and filtered like pt_denoise. Output and pt_postprocess_denoised as pt_denoise.
 * The history, the previous call's guides and its camera belong to the render target: pt_render_begin at the same extent
 * keeps them (a moving camera restarts the accumulation every frame), an extent change, pt_scene_upload, pt_scene_update
 * and pt_texture_upload discard them, and pt_denoise does not touch them. Other changes of the render parameters or of the
 * light-sampling mode are the caller's to handle (with reset = 1). lens_radius > 0 is PT_ERR_UNSUPPORTED; a target holding
 * an adaptive render is PT_ERR_INVALID_ARGUMENT. */
PT_API pt_status pt_denoise_temporal(pt_context *ctx, const pt_render_params *params, const pt_denoise_params *denoise,
                                     const pt_temporal_params *temporal, uint32_t total_samples, float *out_rgba, size_t out_bytes);

/* The history after the last call, per pixel (row-major, `pixels` >= width * height): (integrated irradiance.rgb, history
 * length n) and (m1, m2), the moving averages of the luminance and its square. Either may be NULL. */
PT_API pt_status pt_denoise_temporal_history(pt_context *ctx, float *out_irradiance_n, float *out_moments, size_t pixels);

/* ---- adaptive sampling (DESIGN §3i) --------------------------------------- */

/* Each pixel keeps its sample count and Welford statistics (mean, M2) of its samples' luminance
 * l = (0.2126 r + 0.7152 g) + 0.0722 b.  A pixel is converged when M2 <= t^2 (mean^2 + 0.01) n (n - 1), i.e. the
 * relative standard error of its mean is at most t = threshold.  Pixels move in 8x4 blocks aligned at (0, 0): a block
 * is active while its count is below min_samples, or below max_samples with a pixel that is not converged. */
typedef struct pt_adaptive_params {
    uint32_t min_samples;    /* >= 2: every pixel's samples before its error is first judged           */
    uint32_t max_samples;    /* >= min_samples: per-pixel cap                                          */
    uint32_t batch;          /* >= 1: samples between two judgements                                   */
    uint32_t min_pass_items; /* 0 = 2^21: a pass renders at least this many (pixel, sample) items      */
    float threshold;         /* >= 0, finite: relative standard error at which a block stops           */
} pt_adaptive_params;

typedef struct pt_adaptive_info {
    uint32_t passes;
    uint32_t min_count, max_count;   /* over the frame after the call                              */
    uint32_t unconverged_pixels;     /* pixels that stopped at max_samples without meeting threshold */
    uint64_t samples;                /* (pixel, sample) items rendered by this call                 */
} pt_adaptive_info;

/* Renders until no block is active.  Each pass takes the smallest count n among the active blocks and the next larger
 * one, `next`, and renders samples [n, n + k) of the A pixels of the active blocks at n, with
 * k = min(max_samples, next, max(n + batch, min_samples, n + ceil(min_pass_items / A))) - n.  Sample s of a pixel is the
 * sample s of pt_render_samples (first_sample 0, the whole frame), so a pixel with n samples holds exactly the
 * accumulation of a uniform n-sample render.  A later call on the same target continues with its own parameters (a lower
 * threshold or a higher cap refines further).  A target holds a uniform render or an adaptive one: this call fails with
 * PT_ERR_INVALID_ARGUMENT after pt_render_samples / pt_render_frames wrote to the target, and those fail on a target
 * holding an adaptive render, until pt_render_begin.  pt_stats covers the whole call.  Blocking. */
PT_API pt_status pt_render_adaptive(pt_context *ctx, const pt_render_params *params, const pt_adaptive_params *adaptive,
                                    pt_adaptive_info *out_info /* may be NULL */);

/* Per pixel (row-major, `pixels` >= width * height): the sample count, and (mean luminance, M2). Either pointer may be NULL. */
PT_API pt_status pt_adaptive_readback(pt_context *ctx, uint32_t *out_counts, float *out_mean_m2, size_t pixels);

/* pt_postprocess's chain on the mean image accum / count of an adaptive render (the divisor is 1). */
PT_API pt_status pt_postprocess_adaptive(pt_context *ctx, const pt_postprocess_params *params, uint32_t output_format,
                                         void *out_pixels, size_t out_bytes);

/* pt_denoise's filter on the mean image accum / count of an adaptive render (the divisor is 1); the result is kept for
 * pt_postprocess_denoised like pt_denoise's. */
PT_API pt_status pt_denoise_adaptive(pt_context *ctx, const pt_render_params *params, const pt_denoise_params *denoise,
                                     float *out_rgba, size_t out_bytes);

/* Waits for all queued work of the context. */
PT_API pt_status pt_synchronize(pt_context *ctx);

/* Primary-hit AOV (the information Debug/debugClosestHit.rchit's RenderModePrimitive /
 * Instance / WorldPosition modes visualise, PT/Shaders/Debug/DebugShaderTypes.incl:18-26):
 * traces the pixel-centre primary ray (PT/Shaders/ray.glsl:87-90) of every pixel of a
 * width x height frame and writes width*height pt_hit records (row-major) to host. */
PT_API pt_status pt_first_hit_aov(pt_context *ctx, const pt_render_params *params, uint32_t width,
                                  uint32_t height, pt_hit *out_hits);

/* traceRayEXT for a batch of host rays: closest hit with the alpha-tested any-hit
 * (PT/Shaders/raygen.rgen:68 + anyhit.rahit). */
PT_API pt_status pt_trace_closest(pt_context *ctx, const pt_ray *rays, uint64_t ray_count, pt_hit *out_hits);

/* traceRayEXT with TerminateOnFirstHit + occlusionAnyhit.rahit (PT/Shaders/raygen.rgen:22-34):
 * out_occluded[i] = 1 if anything with alpha >= 1 lies in (tmin, tmax). */
PT_API pt_status pt_trace_occlusion(pt_context *ctx, const pt_ray *rays, uint64_t ray_count,
                                    uint8_t *out_occluded);

PT_API pt_status pt_get_stats(pt_context *ctx, pt_stats *out_stats);

/* Enables (1) / disables (0, default) the per-ray box / triangle / alpha / texel counters of
 * pt_stats for subsequent pt_render_samples calls.  Counting costs a few instructions per node,
 * so timed runs leave it off and the roofline's N_box / N_tri come from a second, identical
 * (deterministic) run with it on.  rays / samples / hits are always counted. */
PT_API pt_status pt_set_traversal_stats(pt_context *ctx, int32_t enable);

/* Enables (1) / disables (0, default) CUDA-event timing of every kernel launch of subsequent
 * pt_render_samples calls, summed per kernel class into pt_stats.kernel_ms (the per-kernel
 * durations the roofline is computed from; events are recorded on the launching stream). */
PT_API pt_status pt_set_kernel_timing(pt_context *ctx, int32_t enable);

/* Scheduling knobs of the wavefront (no reference counterpart; results do not depend on them,
 * bit for bit).  Keys: "pools" (independent sub-wavefronts on separate CUDA streams, 1..8),
 * "slots" (paths in flight, all pools together; takes effect at the next pt_render_begin that
 * changes the extent, or immediately if no target exists), "sort_hits" (0/1: shade hits in triangle
 * order), "sbuf_mb" (sample-buffer budget per round).  The same knobs are read from the
 * environment at pt_context_create: PT_POOLS, PT_SLOTS, PT_SORT_HITS, PT_SBUF_MB. */
PT_API pt_status pt_set_tuning(pt_context *ctx, const char *key, uint64_t value);
/* NOTE: keys that resize the path state ("slots", "pools") reallocate the render target like pt_render_begin does:
 * the accumulated image is reset.  Set them before rendering. */

/* ------------------------------------------------------------------------- */
/* shader unit-test entry point                                              */
/* ------------------------------------------------------------------------- */

/* Modes of pt_test_shading: the eight functions PTT/Shaders/testShading.comp dispatches on
 * (PTT/Shaders/ShadingTestShaderTypes.incl:18-26), the BSDF test (BsdfTestShaderTypes.incl:13)
 * and the remaining units SURVEY §8(a) lists.  Input/output records are arrays of floats. */
enum {
    PT_TEST_GGX_DISTRIBUTION = 0,    /* in: H.xyz, alpha            out: D                         */
    PT_TEST_LAMBDA = 1,              /* in: V.xyz, alpha            out: Lambda                    */
    PT_TEST_GGX_SMITH = 2,           /* in: V.xyz, alpha            out: G1                        */
    PT_TEST_DIELECTRIC_FRESNEL = 3,  /* in: VdotH, eta              out: F                         */
    PT_TEST_SCHLICK_FRESNEL = 4,     /* in: VdotH                   out: F                         */
    PT_TEST_EVALUATE_REFLECTION = 5, /* in: V.xyz, L.xyz, F.xyz, alpha       out: f.xyz, pdf       */
    PT_TEST_EVALUATE_REFRACTION = 6, /* in: V.xyz, L.xyz, F.xyz, alpha, eta  out: f.xyz, pdf       */
    PT_TEST_SAMPLE_GGX = 7,          /* in: u.xy, V.xyz, alpha      out: H.xyz                     */
    PT_TEST_SAMPLE_LOBE_PDFS = 8,    /* in: metalness, transmission, F  out: D, G, M, T            */
    PT_TEST_EVALUATE_BSDF = 9,       /* in: material[17], V.xyz, L.xyz  out: f.xyz, pdf            */
    PT_TEST_SAMPLE_BSDF = 10,        /* in: material[17], V.xyz, rng(bits) out: dir.xyz, pdf, color.xyz, rng(bits) */
    PT_TEST_RNG = 11,                /* in: px, py, width, frame (bits)  out: seed, 4 x state (bits), 4 x float   */
    PT_TEST_PRIMARY_RAY = 12,        /* in: px,py,w,h (bits), u.xy, u2.xy, lens, focal, view_inv[16], proj_inv[16]
                                        out: ray o,d; rx o,d; ry o,d (18 floats)                    */
    PT_TEST_OFFSET_SELF_INTERSECTION = 13, /* in: origin.xyz, normal.xyz   out: p.xyz              */
    PT_TEST_CONCENTRIC_DISK = 14,    /* in: u.xy                     out: d.xy                     */
    PT_TEST_TANGENT_SPACE = 15,      /* in: n.xyz                    out: t.xyz, b.xyz, n.xyz      */
    /* tracing.glsl:2-148, ray.glsl:109-131, sampling.glsl:5-56, material.glsl:55-60, common.glsl:17-20 */
    PT_TEST_DPN_DUV = 16,            /* in: v0, v1, v2 as (position.xyz, uv.xy, normal.xyz), vertex tangent.xyz,
                                        bitangent.xyz (30)            out: dpdu, dpdv, dndu, dndv (12) */
    PT_TEST_DP_DXY = 17,             /* in: p, rxOrigin, rxDirection, ryOrigin, ryDirection, n (18)  out: dpdx, dpdy */
    PT_TEST_DERIVATIVES = 18,        /* in: dpdx, dpdy, dpdu, dpdv (12)   out: dudx, dvdx, dudy, dvdy */
    PT_TEST_REFLECTED_DIFFERENTIALS = 19, /* in: derivatives[4], n, p, viewDir, reflectedDir, dndu, dndv, rxO, rxD,
                                        ryO, ryD (34)                 out: rxO, rxD, ryO, ryD (12)  */
    PT_TEST_REFRACTED_DIFFERENTIALS = 20, /* in: derivatives[4], n, p, viewDir, refractedDir, dndu, dndv, eta, rxO,
                                        rxD, ryO, ryD (35)            out: rxO, rxD, ryO, ryD (12)  */
    PT_TEST_SHADOW_TERMINATOR = 21,  /* in: vertex position, (position, normal) of v0, v1, v2, barycentrics.xyz,
                                        isRefracted (25)              out: origin.xyz               */
    PT_TEST_SAMPLE_LIGHT = 22,       /* in: u.xyz, position.xyz, directional colour.xyz + direction.xyz, one point
                                        light colour.xyz + position.xyz + attenuation c/l/q, light count (bits,
                                        0 or 1) (22)   out: direction.xyz, distance, colour.xyz, attenuation, pdf */
    PT_TEST_TRANSFORM_VERTEX = 23,   /* in: position, normal, tangent, bitangent (12), mesh transform (12: GLSL
                                        mat3x4 = the rows), instance object-to-world (12: rows)
                                        out: position, normal, tangent, bitangent (12)               */
    PT_TEST_RECONSTRUCT_NORMAL = 24, /* in: texel.xyz                out: normal.xyz                */
    PT_TEST_HDR_TO_LDR = 25,         /* in: rgb                      out: rgb                       */
    PT_TEST_MODE_COUNT = 26
};

/* floats per input / output record of each mode (initialiser lists for a uint32_t[PT_TEST_MODE_COUNT]) */
#define PT_TEST_INPUT_STRIDES { 4, 4, 4, 2, 1, 10, 11, 6, 3, 23, 21, 4, 42, 6, 2, 3, 30, 18, 12, 34, 35, 25, 22, 36, 3, 3 }
#define PT_TEST_OUTPUT_STRIDES { 1, 1, 1, 1, 1, 4, 4, 3, 4, 4, 8, 9, 18, 3, 2, 9, 12, 6, 4, 12, 12, 3, 9, 12, 3, 3 }

/* Number of floats per input / output record of a mode (0 for an unknown mode). */
PT_API uint32_t pt_test_input_stride(uint32_t mode);
PT_API uint32_t pt_test_output_stride(uint32_t mode);

/* Replaces TestRenderer::ExecutePipeline("testShading.comp" / "testBsdf.comp", {mode}, N)
 * (PTT/TestRenderer.cpp:79-106): runs the production __device__ function of `mode` on
 * `count` input records in a one-thread-per-record kernel. */
PT_API pt_status pt_test_shading(pt_context *ctx, uint32_t mode, const float *input, float *output,
                                 uint32_t count);

/* ------------------------------------------------------------------------- */
/* debug view (SURVEY §8f rank 4)                                            */
/* ------------------------------------------------------------------------- */

/* PT/Shaders/Debug/DebugShaderTypes.incl:18-42: the specialisation constants of the debug pipeline
 * (Renderer::SetDebugRenderMode / SetDebugRaygenFlags / SetDebugHitGroupFlags). */
enum {
    PT_DEBUG_MODE_COLOR = 0, /* ambient + emissive + raster-style Cook-Torrance direct light with shadow rays */
    PT_DEBUG_MODE_WORLD_POSITION = 1,
    PT_DEBUG_MODE_NORMAL = 2, /* shading normal incl. the normal map */
    PT_DEBUG_MODE_TEXTURE_COORDS = 3,
    PT_DEBUG_MODE_MIPS = 4,   /* 0.1 * lod + 1 */
    PT_DEBUG_MODE_GEOMETRY = 5, /* hashed colours of gl_GeometryIndexEXT / gl_PrimitiveID / gl_InstanceID */
    PT_DEBUG_MODE_PRIMITIVE = 6,
    PT_DEBUG_MODE_INSTANCE = 7
};
enum { PT_DEBUG_RAYGEN_FORCE_OPAQUE = 0x1, PT_DEBUG_RAYGEN_CULL_BACK_FACES = 0x2 /* gl_RayFlagsCullBackFacingTrianglesEXT:
    facing in object space, front = clockwise from the ray origin (Vulkan's default, no instance flags) */ };
enum {
    PT_DEBUG_HIT_DISABLE_COLOR_TEXTURE = 0x01,
    PT_DEBUG_HIT_DISABLE_NORMAL_TEXTURE = 0x02,
    PT_DEBUG_HIT_DISABLE_MIP_MAPS = 0x04,
    PT_DEBUG_HIT_DISABLE_SHADOWS = 0x08,
    PT_DEBUG_HIT_DX_NORMAL_TEXTURES = 0x10
};
typedef struct pt_debug_params {
    uint32_t render_mode;     /* PT_DEBUG_MODE_* */
    uint32_t raygen_flags;    /* PT_DEBUG_RAYGEN_* */
    uint32_t hit_group_flags; /* PT_DEBUG_HIT_* */
} pt_debug_params;

/* Replaces one dispatch of the reference's debug ray-tracing pipeline (Renderer::SetPathTracingPipeline
 * with a debug config; PT/Shaders/Debug/debugRaygen.rgen, debugClosestHit.rchit, debugAnyhit.rahit,
 * debugMiss.rmiss): one pixel-centre ray per pixel, the selected view of the first hit, written as
 * width*height RGBA floats (what the pipeline stores into its rgba32f image) to host memory.
 * params->miss_flags selects the sky like in the path tracer; its other fields besides the camera
 * are unused. */
PT_API pt_status pt_debug_render(pt_context *ctx, const pt_render_params *params, const pt_debug_params *debug,
                                 uint32_t width, uint32_t height, float *out_rgba);

/* Sampler probe: the production texture fetch of one bindless slot (0-8 built in, 9+ scene textures)
 * for `count` records of (uv.xy, dPdx.xy, dPdy.xy).  use_grad = 1: textureGrad as the material
 * fetches use it (PT/Shaders/material.glsl:62-171; sampler of PT/Renderer/Renderer.cpp:103-112:
 * linear / linear-mip / repeat); use_grad = 0: texture() at level 0 as the any-hit and miss stages use
 * it (anyhit.rahit:51, miss.rmiss:27).  Writes count RGBA float4.  The reference has no counterpart
 * (its sampler is hardware); this is the parity hook for the software sampler. */
PT_API pt_status pt_test_texture(pt_context *ctx, uint32_t slot, const float *in6, float *out4, uint32_t count,
                                 int32_t use_grad);

/* Flags of pt_test_trace. */
enum {
    PT_TEST_TRACE_OCCLUSION = 0x1,  /* occlusion query (k_shadow's); otherwise closest hit (k_extend's)          */
    PT_TEST_TRACE_PERSISTENT = 0x2, /* the render's persistent traversal (dynamic ray fetch, straggler splitting);
                                       otherwise the per-thread traversal of pt_trace_closest / pt_trace_occlusion */
    PT_TEST_TRACE_STATS = 0x4       /* the traversal-statistics instantiation, with the tail counters           */
};

/* Traversal probe: traces `ray_count` host rays with the traversal the render's trace kernels run, so that its hits
 * can be compared with the standalone queries hit for hit.  Every ray must have the same tmin (the persistent traversal
 * takes one; PT_ERR_INVALID_ARGUMENT otherwise).  out_hits gets one pt_hit per ray; for occlusion queries
 * instance != PT_NO_HIT means occluded.  out_decals (may be NULL) gets r, g, b, a, dist per ray: the decal record of
 * a closest-hit query on a scene with alpha-tested geometry (dist = -1: none).  blocks = 0 launches the resident grid
 * of the render; a small count (1) sends nearly all rays through the drain mode.  out_tail (may be NULL) gets
 * {warp_iterations, warp_drain_iterations, max_warp_drain_iterations, stack_overflows} (the first three counted with
 * PT_TEST_TRACE_STATS | PT_TEST_TRACE_PERSISTENT only). */
PT_API pt_status pt_test_trace(pt_context *ctx, const pt_ray *rays, uint64_t ray_count, uint32_t flags, uint32_t blocks,
                               pt_hit *out_hits, float *out_decals, uint64_t *out_tail);

#ifdef __cplusplus
}
#endif

#endif /* PT_CORE_H */
