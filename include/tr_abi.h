/* tr_abi.h — the drop-in boundary of the B200-native light-transport path.
 *
 * Plain C ABI (extern "C", pointers + sizes, no torch/CUDA types in the
 * signatures).  Two things live here:
 *
 *  1. the reference's `#[repr(C)]` host<->GPU structs, byte for byte
 *     (/root/reference/shared-structs/src/lib.rs, offsets verified against the
 *     shipped SPIR-V, SURVEY.md Appendix A) — every size/offset is pinned by a
 *     static assert below;
 *  2. the entry points that replace the reference's Vulkan plumbing
 *     (src/render_passes.rs, src/pipelines.rs, src/descriptor_sets.rs) and the
 *     frame recorder `record()` (src/main.rs:1551-2263).  Each export cites
 *     the reference interface it stands in for.
 *
 * All functions return 0 (TR_OK) or a negative tr_status; tr_last_error()
 * gives a thread-local message.  Nothing here ever falls back to a CPU path:
 * if the CUDA device or a kernel is unavailable the call fails.
 */
#ifndef TR_ABI_H
#define TR_ABI_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#define TR_STATIC_ASSERT(c, m) static_assert(c, m)
#else
#define TR_STATIC_ASSERT(c, m) _Static_assert(c, m)
#endif

#define TR_ALIGN16 __attribute__((aligned(16)))
#if defined(_WIN32)
#define TR_API
#else
#define TR_API __attribute__((visibility("default")))
#endif

/* ------------------------------------------------------------------ */
/* glam 0.19 value types (SSE2 layout: Vec4/Quat/Vec3A/Mat4 16-aligned) */
/* ------------------------------------------------------------------ */
typedef struct { float x, y; } tr_vec2;
typedef struct { uint32_t x, y; } tr_uvec2;
typedef struct { float x, y, z; } tr_vec3;
typedef struct TR_ALIGN16 { float x, y, z, w; } tr_vec4;
typedef struct TR_ALIGN16 { float x, y, z, _pad; } tr_vec3a;
typedef struct TR_ALIGN16 { float x, y, z, w; } tr_quat;
typedef struct TR_ALIGN16 { tr_vec4 col[4]; } tr_mat4; /* column-major */

/* ------------------------------------------------------------------ */
/* shared-structs (reference: shared-structs/src/lib.rs)               */
/* ------------------------------------------------------------------ */

/* shared-structs/src/lib.rs:11-16 */
typedef struct TR_ALIGN16 {
    tr_mat4 proj_view;
    tr_vec3a view_position;
    tr_uvec2 framebuffer_size;
    uint64_t acceleration_structure_address; /* 0 = no ray queries, else the handle of tr_build_acceleration_structures */
} tr_push_constants;

/* shared-structs/src/lib.rs:35-41 */
typedef struct {
    float z_near, z_far, scale, bias;
    uint32_t num_depth_slices;
} tr_light_cluster_coefficients;

/* shared-structs/src/lib.rs:21-29 */
typedef struct TR_ALIGN16 {
    tr_light_cluster_coefficients light_clustering_coefficients;
    tr_vec3a sun_dir;
    tr_vec3a sun_intensity;
    tr_vec2 cluster_size_in_pixels;
    tr_uvec2 num_clusters;
    uint32_t debug_clusters;         /* must be 0 */
    uint32_t ggx_lut_texture_index;  /* kept for layout; the LUT is bound by tr_set_ggx_lut */
} tr_uniforms;

/* shared-structs/src/lib.rs:74-78 */
typedef struct TR_ALIGN16 {
    tr_vec4 position_and_spotlight_epsilon;
    tr_vec4 colour_emission_and_falloff_distance_sq;
    tr_vec4 spotlight_direction_and_outer_angle; /* w == 0 => point light */
} tr_light;

/* shared-structs/src/lib.rs:143-153 */
typedef struct {
    int32_t diffuse, metallic_roughness, normal_map, emissive, occlusion,
        transmission, thickness, specular, specular_colour; /* -1 = none */
} tr_textures;

/* shared-structs/src/lib.rs:157-173 */
typedef struct TR_ALIGN16 {
    tr_textures textures;
    float metallic_factor;
    float roughness_factor;
    float alpha_clipping_cutoff;
    tr_vec4 diffuse_factor;
    tr_vec3a emissive_factor;
    float normal_map_scale;
    float occlusion_strength;
    float index_of_refraction;
    float transmission_factor;
    float thickness_factor;
    float attenuation_distance;
    tr_vec3a attenuation_colour;
    float specular_factor;
    tr_vec3a specular_colour_factor;
} tr_material_info;

/* shared-structs/src/lib.rs:178-181 */
typedef struct TR_ALIGN16 {
    tr_vec4 translation_and_scale; /* w = uniform scale */
    tr_quat rotation;
} tr_packed_similarity;

/* shared-structs/src/lib.rs:253-257 */
typedef struct TR_ALIGN16 {
    tr_packed_similarity transform;
    uint32_t primitive_id;
    uint32_t material_id;
} tr_instance;

/* shared-structs/src/lib.rs:262-268 */
typedef struct TR_ALIGN16 {
    tr_vec4 packed_bounding_sphere; /* xyz centre, w radius, model space */
    uint32_t draw_buffer_index;     /* 0 opaque, 1 alpha clip, 2 transmission, 3 transmission alpha clip (model_loading.rs:68-78) */
    uint32_t index_count;
    uint32_t first_index;
    uint32_t first_instance;
} tr_primitive_info;

/* shared-structs/src/lib.rs:273-280 */
typedef struct TR_ALIGN16 {
    tr_mat4 view;
    tr_vec2 frustum_x_xz;
    tr_vec2 frustum_y_yz;
    float z_near;
} tr_culling_push_constants;

/* shared-structs/src/lib.rs:285-288 */
typedef struct TR_ALIGN16 {
    tr_vec3a min;
    tr_vec3a max;
} tr_cluster_aabb;

/* shared-structs/src/lib.rs:336-339 */
typedef struct TR_ALIGN16 {
    tr_mat4 inverse_perspective;
    tr_uvec2 screen_dimensions;
} tr_write_cluster_data_push_constants;

/* shared-structs/src/lib.rs:344-347 */
typedef struct TR_ALIGN16 {
    tr_mat4 view_matrix;
    tr_quat view_rotation;
} tr_assign_lights_push_constants;

/* shader/src/lib.rs:401-409 (vk::DrawIndexedIndirectCommand) */
typedef struct {
    uint32_t index_count;
    uint32_t instance_count;
    uint32_t first_index;
    int32_t vertex_offset;
    uint32_t first_instance;
} tr_draw_indexed_indirect_command;

/* shader/src/tonemapping.rs:28-38 */
typedef struct {
    float a, b, c, d, crosstalk, saturation, cross_saturation;
} tr_baked_lottes_tonemapper_params;

#define TR_MAX_LIGHTS_PER_CLUSTER 128u /* shared-structs/src/lib.rs:322 */
#define TR_NUM_DRAW_BUFFERS 4u         /* shader/src/lib.rs:471 */

TR_STATIC_ASSERT(sizeof(tr_push_constants) == 96, "PushConstants");
TR_STATIC_ASSERT(offsetof(tr_push_constants, view_position) == 64, "PushConstants.view_position");
TR_STATIC_ASSERT(offsetof(tr_push_constants, framebuffer_size) == 80, "PushConstants.framebuffer_size");
TR_STATIC_ASSERT(offsetof(tr_push_constants, acceleration_structure_address) == 88, "PushConstants.as_address");
TR_STATIC_ASSERT(sizeof(tr_light_cluster_coefficients) == 20, "LightClusterCoefficients");
TR_STATIC_ASSERT(sizeof(tr_uniforms) == 96, "Uniforms");
TR_STATIC_ASSERT(offsetof(tr_uniforms, sun_dir) == 32, "Uniforms.sun_dir");
TR_STATIC_ASSERT(offsetof(tr_uniforms, sun_intensity) == 48, "Uniforms.sun_intensity");
TR_STATIC_ASSERT(offsetof(tr_uniforms, cluster_size_in_pixels) == 64, "Uniforms.cluster_size_in_pixels");
TR_STATIC_ASSERT(offsetof(tr_uniforms, num_clusters) == 72, "Uniforms.num_clusters");
TR_STATIC_ASSERT(offsetof(tr_uniforms, debug_clusters) == 80, "Uniforms.debug_clusters");
TR_STATIC_ASSERT(offsetof(tr_uniforms, ggx_lut_texture_index) == 84, "Uniforms.ggx_lut_texture_index");
TR_STATIC_ASSERT(sizeof(tr_light) == 48, "Light");
TR_STATIC_ASSERT(sizeof(tr_textures) == 36, "Textures");
TR_STATIC_ASSERT(sizeof(tr_material_info) == 160, "MaterialInfo");
TR_STATIC_ASSERT(offsetof(tr_material_info, metallic_factor) == 36, "MaterialInfo.metallic_factor");
TR_STATIC_ASSERT(offsetof(tr_material_info, roughness_factor) == 40, "MaterialInfo.roughness_factor");
TR_STATIC_ASSERT(offsetof(tr_material_info, alpha_clipping_cutoff) == 44, "MaterialInfo.alpha_clipping_cutoff");
TR_STATIC_ASSERT(offsetof(tr_material_info, diffuse_factor) == 48, "MaterialInfo.diffuse_factor");
TR_STATIC_ASSERT(offsetof(tr_material_info, emissive_factor) == 64, "MaterialInfo.emissive_factor");
TR_STATIC_ASSERT(offsetof(tr_material_info, normal_map_scale) == 80, "MaterialInfo.normal_map_scale");
TR_STATIC_ASSERT(offsetof(tr_material_info, occlusion_strength) == 84, "MaterialInfo.occlusion_strength");
TR_STATIC_ASSERT(offsetof(tr_material_info, index_of_refraction) == 88, "MaterialInfo.index_of_refraction");
TR_STATIC_ASSERT(offsetof(tr_material_info, transmission_factor) == 92, "MaterialInfo.transmission_factor");
TR_STATIC_ASSERT(offsetof(tr_material_info, thickness_factor) == 96, "MaterialInfo.thickness_factor");
TR_STATIC_ASSERT(offsetof(tr_material_info, attenuation_distance) == 100, "MaterialInfo.attenuation_distance");
TR_STATIC_ASSERT(offsetof(tr_material_info, attenuation_colour) == 112, "MaterialInfo.attenuation_colour");
TR_STATIC_ASSERT(offsetof(tr_material_info, specular_factor) == 128, "MaterialInfo.specular_factor");
TR_STATIC_ASSERT(offsetof(tr_material_info, specular_colour_factor) == 144, "MaterialInfo.specular_colour_factor");
TR_STATIC_ASSERT(sizeof(tr_packed_similarity) == 32, "PackedSimilarity");
TR_STATIC_ASSERT(sizeof(tr_instance) == 48, "Instance");
TR_STATIC_ASSERT(offsetof(tr_instance, primitive_id) == 32, "Instance.primitive_id");
TR_STATIC_ASSERT(offsetof(tr_instance, material_id) == 36, "Instance.material_id");
TR_STATIC_ASSERT(sizeof(tr_primitive_info) == 32, "PrimitiveInfo");
TR_STATIC_ASSERT(offsetof(tr_primitive_info, draw_buffer_index) == 16, "PrimitiveInfo.draw_buffer_index");
TR_STATIC_ASSERT(sizeof(tr_culling_push_constants) == 96, "CullingPushConstants");
TR_STATIC_ASSERT(offsetof(tr_culling_push_constants, frustum_x_xz) == 64, "CullingPushConstants.frustum_x_xz");
TR_STATIC_ASSERT(offsetof(tr_culling_push_constants, frustum_y_yz) == 72, "CullingPushConstants.frustum_y_yz");
TR_STATIC_ASSERT(offsetof(tr_culling_push_constants, z_near) == 80, "CullingPushConstants.z_near");
TR_STATIC_ASSERT(sizeof(tr_cluster_aabb) == 32, "ClusterAabb");
TR_STATIC_ASSERT(sizeof(tr_write_cluster_data_push_constants) == 80, "WriteClusterDataPushConstants");
TR_STATIC_ASSERT(offsetof(tr_write_cluster_data_push_constants, screen_dimensions) == 64, "WriteClusterData.screen_dimensions");
TR_STATIC_ASSERT(sizeof(tr_assign_lights_push_constants) == 80, "AssignLightsPushConstants");
TR_STATIC_ASSERT(offsetof(tr_assign_lights_push_constants, view_rotation) == 64, "AssignLights.view_rotation");
TR_STATIC_ASSERT(sizeof(tr_draw_indexed_indirect_command) == 20, "DrawIndexedIndirectCommand");
TR_STATIC_ASSERT(sizeof(tr_baked_lottes_tonemapper_params) == 28, "BakedLottesTonemapperParams");

/* ------------------------------------------------------------------ */
/* glam-pbr batch contracts (reference: glam-pbr/src/lib.rs)           */
/* SoA-free "array of params" form of the pub fns; Rust closures cannot */
/* cross a C ABI so the samplers are data (pyramid + LUT bound on ctx). */
/* ------------------------------------------------------------------ */

/* glam-pbr/src/lib.rs:171-179 MaterialParams */
typedef struct {
    tr_vec3 diffuse_colour;
    float metallic;
    float perceptual_roughness;
    float index_of_refraction;
    tr_vec3 specular_colour;
    float specular_factor;
} tr_material_params;

/* glam-pbr/src/lib.rs:163-169 BasicBrdfParams */
typedef struct {
    tr_vec3 normal;
    tr_vec3 light;
    tr_vec3 light_intensity;
    tr_vec3 view;
    tr_material_params material_params;
} tr_basic_brdf_params;

/* glam-pbr/src/lib.rs:437-441 BrdfResult */
typedef struct {
    tr_vec3 diffuse;
    tr_vec3 specular;
} tr_brdf_result;

/* glam-pbr/src/lib.rs:200-205 arguments of transmission_btdf */
typedef struct {
    tr_material_params material_params;
    tr_vec3 normal;
    tr_vec3 view;
    tr_vec3 light;
} tr_transmission_btdf_params;

/* glam-pbr/src/lib.rs:235-246 IblVolumeRefractionParams (proj_view_matrix passed once per batch) */
typedef struct {
    tr_material_params material_params;
    uint32_t framebuffer_size_x;
    tr_vec3 normal;
    tr_vec3 view;
    tr_vec3 position;
    float thickness;
    float model_scale;
    float attenuation_distance;
    tr_vec3 attenuation_colour;
} tr_ibl_volume_refraction_params;

/* One iteration of the clustered-light loops for a point light — shader/src/lighting.rs:179-216 (`evaluate_lights`) and
 * :58-92 (`evaluate_lights_transmission`): light_direction_and_attenuation(position, light_position) (glam-pbr
 * lib.rs:12-23), then basic_brdf(normal, direction, colour * attenuation, view, material) and
 * transmission_btdf(material, normal, view, direction) * colour * attenuation.  `normal` and `view` are unit vectors
 * (the shaders normalise them before the loop).  tr_eval_point_light runs the SAME device code as the frame kernels'
 * light loop (fast regime + adaptive exactness), so the hot loop has a per-element contract test of its own. */
typedef struct {
    tr_vec3 normal;
    tr_vec3 view;
    tr_vec3 position;       /* fragment, world space */
    tr_vec3 light_position;
    tr_vec3 light_colour;   /* Light::colour_emission (rgb = colour * intensity) */
    tr_material_params material_params;
} tr_point_light_params;

typedef struct {
    tr_vec3 diffuse;        /* BrdfResult.diffuse */
    tr_vec3 specular;       /* BrdfResult.specular */
    tr_vec3 transmission;   /* transmission_btdf(..) * light */
} tr_point_light_result;

TR_STATIC_ASSERT(sizeof(tr_material_params) == 40, "MaterialParams (C form)");
TR_STATIC_ASSERT(sizeof(tr_point_light_params) == 100, "point-light loop iteration params");
TR_STATIC_ASSERT(sizeof(tr_point_light_result) == 36, "point-light loop iteration result");
TR_STATIC_ASSERT(sizeof(tr_basic_brdf_params) == 88, "BasicBrdfParams (C form)");
TR_STATIC_ASSERT(sizeof(tr_transmission_btdf_params) == 76, "transmission_btdf params (C form)");
TR_STATIC_ASSERT(sizeof(tr_ibl_volume_refraction_params) == 104, "IblVolumeRefractionParams (C form)");

/* ------------------------------------------------------------------ */
/* Status, config, opaque context                                       */
/* ------------------------------------------------------------------ */
typedef enum {
    TR_OK = 0,
    TR_ERR_INVALID_ARG = -1,
    TR_ERR_UNSUPPORTED = -2, /* e.g. debug_clusters != 0 */
    TR_ERR_CUDA = -3,
    TR_ERR_NCCL = -4,
    TR_ERR_OOM = -5,
    TR_ERR_STATE = -6 /* call order violated (e.g. shade before a G-buffer exists) */
} tr_status;

typedef struct tr_ctx tr_ctx;

typedef struct {
    uint32_t width, height;  /* full framebuffer size (main.rs: extent) */
    int32_t device;          /* CUDA ordinal */
    uint32_t band_y0, band_y1; /* rows this context shades; y1 == 0 => whole frame */
    uint32_t flags;          /* TR_FLAG_* */
} tr_config;

#define TR_FLAG_HDR_F32_DEBUG 1u /* also keep an fp32 copy of the HDR target (parity tests) */

/* G-buffer planes (structure-of-arrays, one element per pixel, row-major,
 * row stride = width).  This is what the reference's rasteriser hands the
 * fragment stage as varyings (shader/src/lib.rs:37-56,164-181), flattened:
 *   depth        frag_coord.z (reversed-Z, 0 = empty pixel; main.rs:1586-1591)
 *   normal       interpolated `rotation * normal` (un-normalised, lib.rs:356)
 *   uv           interpolated uv (lib.rs:357)
 *   material_id  flat (lib.rs:358)
 *   scale        flat similarity.scale (transmissive layer only, lib.rs:388)
 *   position     optional explicit world position; NULL => reconstructed from
 *                depth and the pixel centre with inverse(proj_view)
 */
typedef struct {
    const float* depth;          /* [h*w]   */
    const float* normal;         /* [h*w*3] */
    const float* uv;             /* [h*w*2] */
    const uint32_t* material_id; /* [h*w]   */
    const float* scale;          /* [h*w] or NULL (layer 0) */
    const float* position;       /* [h*w*3] or NULL */
    /* forward differences to the right / lower neighbour on the pixel's own triangle: what the 2x2 quad gives the
     * reference's fragment stage implicitly (texture level of detail; ddx/ddy in lighting.rs:246-249).  NULL => 0. */
    const float* duv;            /* [h*w*4] du/dx, dv/dx, du/dy, dv/dy */
    const float* ddepth;         /* [h*w*2] d(frag_coord.z)/dx, /dy */
} tr_gbuffer_planes;

typedef struct {
    float* depth;
    float* normal;
    float* uv;
    uint32_t* material_id;
    float* scale;
    float* position; /* filled only if the layer carries explicit positions */
    float* duv;      /* filled only once textures are bound (tr_set_texture) */
    float* ddepth;
} tr_gbuffer_planes_out;

enum { TR_LAYER_OPAQUE = 0, TR_LAYER_TRANSMISSIVE = 1 };

/* ------------------------------------------------------------------ */
/* Lifecycle — replaces Pipelines::new / DescriptorSets::allocate       */
/* (src/pipelines.rs:46-172, src/descriptor_sets.rs:150-316) and the    */
/* LoopDestroyed cleanup (src/main.rs:1416-1445).                        */
/* ------------------------------------------------------------------ */
TR_API int32_t tr_create(const tr_config* config, tr_ctx** out_ctx);
TR_API int32_t tr_destroy(tr_ctx* ctx);
/* swapchain-resize path, src/main.rs:996-1166: reallocates depth/hdr/pyramid. */
TR_API int32_t tr_resize(tr_ctx* ctx, uint32_t width, uint32_t height);
TR_API int32_t tr_set_band(tr_ctx* ctx, uint32_t y0, uint32_t y1);
TR_API const char* tr_last_error(void);
TR_API const char* tr_version(void);
/* Run every subsequent call on this CUDA stream (a cudaStream_t cast to void*; NULL = the context's own). */
TR_API int32_t tr_set_stream(tr_ctx* ctx, void* cuda_stream);
/* fence wait, src/main.rs:1290 */
TR_API int32_t tr_sync(tr_ctx* ctx);

/* ------------------------------------------------------------------ */
/* Uploads — replace the descriptor writes, src/main.rs:715-828         */
/* ------------------------------------------------------------------ */
/* Device sources.  tr_set_lights, tr_update_mesh_vertices and tr_update_instance_transforms also take their arrays in device
 * memory (the context's device, another device, or managed memory), so a pose or a light set computed on the GPU goes in
 * without a copy through the host.  A device source is read on the context stream at the point of the call: its producer
 * must be ordered before that point, either by running on the context stream (tr_set_stream) or by an event the caller
 * makes the context stream wait for.  It may be reused once the context stream has passed the call.  None of these calls
 * waits for the device, and none allocates except when a buffer grows.  The members of a group are updated one by one, as
 * for the other uploads; a source on another device of the group is read with the same copy. */
TR_API int32_t tr_set_instances(tr_ctx* ctx, const tr_instance* instances, uint32_t n);      /* set1/b0, main.rs:2527 */
/* The instance write of --rotate-model (src/main.rs:1263-1345) for instances whose ids do not change: replaces the transform of
 * instances [first, first + n) and keeps their primitive_id and material_id, so unlike tr_set_instances it needs no host copy
 * of the records.  The source may be pageable, page-locked or device memory (see "Device sources"); a host source is copied
 * into a staging buffer of the context first (grow-only), a device one is read in place.  Stream-ordered on the context
 * stream: the frame enqueued before the call sees the old transforms, the next one the new.  As after tr_set_instances, a
 * traced frame then fails with TR_ERR_STATE until tr_update_top_level_acceleration_structure(_async) has run.  Non-finite
 * values are accepted.  Errors: a range past the instance count, or a null pointer with n > 0: TR_ERR_INVALID_ARG; a rejected
 * call changes nothing; n = 0: nothing.  Each call launches 1 kernel (tr_launch_count). */
TR_API int32_t tr_update_instance_transforms(tr_ctx* ctx, uint32_t first, uint32_t n, const tr_packed_similarity* transforms);
TR_API int32_t tr_set_primitives(tr_ctx* ctx, const tr_primitive_info* prims, uint32_t n);   /* set0/b7 + cull set/b0 */
TR_API int32_t tr_set_materials(tr_ctx* ctx, const tr_material_info* materials, uint32_t n); /* set0/b2 */
/* Host sources follow the upload rule (pageable: copied during the call; page-locked: read in stream order, ahead of the
 * frame in flight, see INTEGRATION.md section 3).  A device source is copied on the context stream (see "Device sources"); of
 * two calls before one frame, host or device in either order, the later one wins. */
TR_API int32_t tr_set_lights(tr_ctx* ctx, const tr_light* lights, uint32_t n);               /* set2/b0, main.rs:472-478 */
TR_API int32_t tr_set_uniforms(tr_ctx* ctx, const tr_uniforms* uniforms);                    /* set0/b3, main.rs:1231 */
/* set0/b0[ggx_lut_texture_index]: RGBA8 UNORM, one mip (main.rs:295-330). */
TR_API int32_t tr_set_ggx_lut(tr_ctx* ctx, const uint8_t* rgba8, uint32_t width, uint32_t height);
/* set0/b0[index]: one bindless sampled image of the material system (src/descriptor_sets.rs, MAX_IMAGES = 193,
 * src/main.rs:59), as the loader creates it (src/model_loading.rs:340-379): RGBA8, `srgb` != 0 for R8G8B8A8_SRGB, with
 * its mip chain.  levels[k] points to mip k, which is max(1, width >> k) x max(1, height >> k) texels, tightly packed.
 * Sampled with the repeat sampler (linear min/mag/mip, src/main.rs:683-692). */
#define TR_MAX_IMAGES 193u
TR_API int32_t tr_set_texture(tr_ctx* ctx, uint32_t index, const uint8_t* const* levels, uint32_t n_levels,
                              uint32_t width, uint32_t height, int32_t srgb);
/* load_texture_from_gltf + ImageManager::push_image (src/model_loading.rs:340-379): level 0 only, as RGBA8 (sRGB when
 * srgb != 0); levels 1 .. n_levels-1 are built on the device in stream order. n_levels = 0 means the full chain
 * floor(log2(min(w, h))) + 1.
 * Each level is the 2x2 box of the one above it (odd sizes cropped to even), filtered in linear light in float64 and rounded
 * back to RGBA8 bytes, as the Python ingest's scenes.make_mips does: the image samples bit for bit as tr_set_texture fed
 * that chain.  Stream-ordered on the context stream: the frame enqueued before the call samples the old image, the next one
 * the new.  The source follows the upload rule (pageable: copied during the call; page-locked: read in stream order).  With
 * a page-locked source the call does not wait for the device, except when `index` is bound and its allocation must grow
 * (as tr_set_texture, it then waits for the frame in flight); binding an index for the first time never waits.  The
 * image's allocation keeps the RGBA8 bytes of its levels beside the decoded texels (+25 %).  tr_set_texture and this call
 * may rebind the same index in any order.  Errors: those of tr_set_texture (index >= TR_MAX_IMAGES, a null pointer, a zero
 * size, n_levels > 16), and n_levels greater than the full chain: TR_ERR_INVALID_ARG; a rejected call changes nothing.
 * Each call launches n_levels kernels (the full chain's count for 0) (tr_launch_count). */
TR_API int32_t tr_set_texture_async(tr_ctx* ctx, uint32_t index, const uint8_t* rgba8, uint32_t width, uint32_t height,
                                    int32_t srgb, uint32_t n_levels);
/* Parity hook: level `level` of bound image `index` as the samplers read it (RGBA32F, max(1, w >> level) x
 * max(1, h >> level) texels, into *w / *h; null array: size only); blocking.  Not bound: TR_ERR_STATE. */
TR_API int32_t tr_read_texture_level(tr_ctx* ctx, uint32_t index, uint32_t level, float* rgba32f, uint32_t* w, uint32_t* h);
/* vertex bindings 0..2 + index buffer (pipelines.rs:291-307, main.rs:2516-2557). */
TR_API int32_t tr_set_mesh(tr_ctx* ctx, const float* positions, const float* normals, const float* uvs,
                           uint32_t n_vertices, const uint32_t* indices, uint32_t n_indices);
/* Vertex animation (skinning, morph targets, cloth, procedural displacement computed on the host or the GPU): replaces the
 * positions and normals [n*3] of vertices [first_vertex, first_vertex + n) of the mesh of tr_set_mesh; indices, uvs and the
 * vertex count stay.  Stream-ordered on the context stream: the frame enqueued before the call sees the old vertices, the next
 * one the new.  Host sources follow the upload rule (pageable: copied during the call; page-locked: read in stream order);
 * device sources are read in stream order too (see "Device sources"); each pointer is classified on its own.  On the device, in
 * stream order, it recomputes the culling spheres of the binning pass and, once tr_build_acceleration_structures has run,
 * refits the bottom-level structures (same topology, new boxes and triangles); the top level then needs an update
 * (tr_update_top_level_acceleration_structure(_async)) before the next traced frame, which otherwise fails with
 * TR_ERR_STATE, as after tr_set_instances.  The handle does not change.  No wait for the device.  No allocation either,
 * except in the first call after tr_set_mesh / tr_set_primitives when no tr_cull has run since: that call sizes the
 * culling-sphere buffers for the new chunk count (grow-only), as the next tr_cull would.
 * PrimitiveInfo.packed_bounding_sphere stays the caller's: for a deforming mesh it must hold every pose.
 * No mesh: TR_ERR_STATE; a range past the vertex count, or a null pointer with n > 0: TR_ERR_INVALID_ARG; n = 0: nothing.
 * Each call launches 1 kernel, plus 2 with built acceleration structures (tr_launch_count). */
TR_API int32_t tr_update_mesh_vertices(tr_ctx* ctx, uint32_t first_vertex, uint32_t n, const float* positions, const float* normals);
/* Parity hook: the culling spheres of the binning pass, one float4 (object-space centre xyz, radius w) per 64 consecutive
 * triangles of every primitive, primitive after primitive; computed first if no tr_cull has needed them yet.  *n_spheres
 * receives the count (0 when a primitive leaves the index buffer: the test is off); null array: count only; blocking. */
TR_API int32_t tr_read_chunk_spheres(tr_ctx* ctx, float* spheres, uint32_t capacity, uint32_t* n_spheres);

/* ------------------------------------------------------------------ */
/* Ray-queried shadows — the `--ray-tracing` option (src/main.rs:84,   */
/* 577-658) and the RayQueryKHR variant of the fragment shaders          */
/* (shader/src/lighting.rs:22-32, 64-71, 97-125, 154-165, 186-195).      */
/* ------------------------------------------------------------------ */
/* build_acceleration_structures_from_primitives + build_top_level_acceleration_structure_from_instances
 * (src/acceleration_structures.rs:6-186, called at src/main.rs:594-649): one bottom-level structure per primitive
 * over the bound mesh, one top-level structure over the bound instances whose primitive has draw_buffer_index < 2
 * (src/main.rs:614-625).  *address is what the reference puts in PushConstants.acceleration_structure_address
 * (src/main.rs:856-859); passing it to tr_frame / tr_shade_* turns the shadow rays on, 0 leaves them off.
 * Rebinding the mesh or the primitives invalidates it. */
TR_API int32_t tr_build_acceleration_structures(tr_ctx* ctx, uint64_t* address);
/* build_acceleration_structures_from_primitives + build_top_level_acceleration_structure_from_instances
 * (src/acceleration_structures.rs:6-186), built on the device in stream order: the contract of
 * tr_build_acceleration_structures (same handle rules, errors, invalidation and read-back hooks), but it reads the
 * positions, indices and instances as the context stream sees them (it may follow tr_set_mesh, tr_update_mesh_vertices or
 * tr_set_instances directly), never waits for the device and allocates only when a buffer grows.  The trees differ from
 * the host build's (H-PLOC, single-triangle leaves: 64 B of nodes per triangle); every ray's result does not.  After
 * refits, it is the cheap rebuild from the current pose. */
TR_API int32_t tr_build_acceleration_structures_async(tr_ctx* ctx, uint64_t* address);
/* update_top_level_acceleration_structure_from_instances (src/acceleration_structures.rs:188-263, src/main.rs:1332-1345):
 * after tr_set_instances.  The handle may change; it is returned again. */
TR_API int32_t tr_update_top_level_acceleration_structure(tr_ctx* ctx, uint64_t* address);
/* update_top_level_acceleration_structure_from_instances (src/acceleration_structures.rs:188-263, src/main.rs:1332-1345),
 * built on the device in stream order: it reads the instance buffer as the context's stream sees it (after any pending
 * tr_set_instances upload) and returns without waiting for the GPU.  The frame enqueued next traces against it.  Same
 * handle rules as tr_update_top_level_acceleration_structure; the handle changes only when the number of instances
 * in the top level grows past what was allocated.  Requires tr_build_acceleration_structures since the last mesh /
 * primitive upload.  A call does not wait for the device unless a buffer grows.  Each call launches 19 kernels
 * (tr_launch_count). */
TR_API int32_t tr_update_top_level_acceleration_structure_async(tr_ctx* ctx, uint64_t* address);
/* trace_shadow_ray (lighting.rs:97-125) for a batch of rays given in host memory: origins/directions [n*3], t_max [n];
 * lit[i] = 1 when nothing is hit between t_min = 0.001 and t_max[i], else 0. */
TR_API int32_t tr_trace_shadow_rays(tr_ctx* ctx, uint32_t n, const float* origins, const float* directions,
                                    const float* t_max, uint8_t* lit);
/* Parity hook: the occluded-ray bits the last shading pass of `layer` used, [5][h*w] words (band rows are written):
 * planes 0-3 bit i = the ray towards the i-th light of the pixel's cluster list, plane 4 bit 0 = the sun ray. */
TR_API int32_t tr_read_shadow_mask(tr_ctx* ctx, int32_t layer, uint32_t* mask);
/* Parity hook: the top level as built, by either update: node_capacity 64-byte nodes and instance_capacity 64-byte
 * instance records in leaf order (layouts in csrc/tr_device_accel.cuh: AccelNode, AccelInstance); node 0 is the root.
 * *n_nodes / *n_instances receive the counts (null arrays: counts only); blocking. */
TR_API int32_t tr_read_top_level_acceleration_structure(tr_ctx* ctx, void* nodes, uint32_t node_capacity, uint32_t* n_nodes,
                                                       void* instances, uint32_t instance_capacity, uint32_t* n_instances);
/* Parity hook: the bottom-level structures of every primitive, as built or as refitted by tr_update_mesh_vertices:
 * node_capacity 64-byte nodes (AccelNode; the trees one after the other in primitive order, each root first) and
 * tri_capacity triangles of three float4 (x, y, z, 0) each, in leaf order, primitive after primitive.  Leaf references
 * count triangles from the first triangle of their primitive.  Counts into *n_nodes / *n_tris (null arrays: counts only);
 * blocking. */
TR_API int32_t tr_read_bottom_level_acceleration_structures(tr_ctx* ctx, void* nodes, uint32_t node_capacity, uint32_t* n_nodes,
                                                           void* tris, uint32_t tri_capacity, uint32_t* n_tris);

/* ------------------------------------------------------------------ */
/* Per-frame passes, in record() order (src/main.rs:1551-2263).        */
/* All enqueue on the context stream and return without blocking.       */
/* ------------------------------------------------------------------ */
/* frustum_culling + demultiplex_draws (shader/src/lib.rs:411-517; dispatch main.rs:1669-1838).
 * Produces instance_counts[n_prim], an ascending visible-instance list,
 * the four draw lists (ascending primitive id) and draw_counts[4]. */
TR_API int32_t tr_cull(tr_ctx* ctx, const tr_culling_push_constants* pc);
/* write_cluster_data (shader/src/lib.rs:519-594; recorded at init/resize, main.rs:1459-1517). */
TR_API int32_t tr_build_clusters(tr_ctx* ctx, const tr_write_cluster_data_push_constants* pc);
/* assign_lights_to_clusters (shader/src/lib.rs:596-645; main.rs:1766-1798); lists come out in ascending light id. */
TR_API int32_t tr_assign_lights(tr_ctx* ctx, const tr_assign_lights_push_constants* pc);
/* depth pre-passes + varyings of both layers (lib.rs:319-391; main.rs:1900-1944, 2005-2042),
 * as a software visibility pass over the culled draw lists. */
TR_API int32_t tr_visibility(tr_ctx* ctx, const tr_push_constants* pc);
/* `fragment` (lib.rs:164-249) over the opaque layer, band rows only. */
TR_API int32_t tr_shade_opaque(tr_ctx* ctx, const tr_push_constants* pc);
/* multi-GPU only: exchange opaque bands so every rank holds the whole mip-0 frame. */
TR_API int32_t tr_allgather_opaque(tr_ctx* ctx);
/* generate_mips (main.rs:2054-2063; level count main.rs:2590-2592). */
TR_API int32_t tr_generate_mips(tr_ctx* ctx);
/* `fragment_transmission` (lib.rs:37-162) over the transmissive layer, band rows only. */
TR_API int32_t tr_shade_transmission(tr_ctx* ctx, const tr_push_constants* pc);
/* fragment_tonemap (lib.rs:683-697, tonemapping.rs) -> sRGB8 RGBA. */
TR_API int32_t tr_tonemap(tr_ctx* ctx, const tr_baked_lottes_tonemapper_params* params);

/* One call = one record(): cull -> assign lights -> visibility -> opaque ->
 * [all-gather] -> mips -> transmission -> tonemap (src/main.rs:1551-2263). */
typedef struct {
    tr_culling_push_constants culling;
    tr_assign_lights_push_constants assign_lights;
    tr_push_constants push_constants;
    tr_baked_lottes_tonemapper_params tonemap;
    uint32_t flags; /* TR_FRAME_* */
} tr_frame_params;
#define TR_FRAME_SKIP_TONEMAP 1u
#define TR_FRAME_SKIP_VISIBILITY 2u /* reuse the injected / previous G-buffer */
TR_STATIC_ASSERT(sizeof(tr_frame_params) == 304, "tr_frame_params");
TR_STATIC_ASSERT(offsetof(tr_frame_params, assign_lights) == 96, "tr_frame_params.assign_lights");
TR_STATIC_ASSERT(offsetof(tr_frame_params, push_constants) == 176, "tr_frame_params.push_constants");
TR_STATIC_ASSERT(offsetof(tr_frame_params, tonemap) == 272, "tr_frame_params.tonemap");
TR_STATIC_ASSERT(offsetof(tr_frame_params, flags) == 300, "tr_frame_params.flags");
TR_API int32_t tr_frame(tr_ctx* ctx, const tr_frame_params* params);
/* Marks the start of a frame for the per-pass timers when the passes are called one by one instead of through tr_frame
 * (the reference collects its per-pass timestamp queries once per frame, src/profiling.rs:101-131). */
TR_API int32_t tr_begin_frame(tr_ctx* ctx);

/* ------------------------------------------------------------------ */
/* Parity hooks: inject / read back every intermediate                  */
/* ------------------------------------------------------------------ */
TR_API int32_t tr_set_gbuffer(tr_ctx* ctx, int32_t layer, const tr_gbuffer_planes* planes);
TR_API int32_t tr_read_gbuffer(tr_ctx* ctx, int32_t layer, const tr_gbuffer_planes_out* planes);
/* mip 0 of the sampled opaque pyramid, RGBA16F bits, full frame. */
TR_API int32_t tr_set_opaque_frame(tr_ctx* ctx, const uint16_t* rgba16f);
/* hdr_framebuffer, RGBA16F bits, full frame (e.g. to tonemap a caller-provided image). */
TR_API int32_t tr_set_hdr(tr_ctx* ctx, const uint16_t* rgba16f);
TR_API int32_t tr_set_cluster_lights(tr_ctx* ctx, const uint32_t* counts, const uint32_t* indices); /* [n_clusters], [n_clusters*128] */
TR_API int32_t tr_read_visible_instances(tr_ctx* ctx, uint32_t* ids, uint32_t capacity, uint32_t* n_visible);
TR_API int32_t tr_read_instance_counts(tr_ctx* ctx, uint32_t* counts, uint32_t capacity);
TR_API int32_t tr_read_draws(tr_ctx* ctx, uint32_t bucket, tr_draw_indexed_indirect_command* cmds,
                             uint32_t capacity, uint32_t* n_draws);
TR_API int32_t tr_read_cluster_aabbs(tr_ctx* ctx, tr_cluster_aabb* aabbs, uint32_t capacity);
TR_API int32_t tr_read_cluster_lights(tr_ctx* ctx, uint32_t* counts, uint32_t* indices); /* [n_clusters], [n_clusters*128] */
TR_API int32_t tr_read_hdr(tr_ctx* ctx, uint16_t* rgba16f);              /* hdr_framebuffer, full frame */
TR_API int32_t tr_read_hdr_f32(tr_ctx* ctx, float* rgba32f);             /* needs TR_FLAG_HDR_F32_DEBUG */
TR_API int32_t tr_read_pyramid_level(tr_ctx* ctx, uint32_t level, uint16_t* rgba16f, uint32_t* w, uint32_t* h);
TR_API int32_t tr_read_srgb8(tr_ctx* ctx, uint8_t* rgba8);
/* Same band copy, enqueued on a copy stream behind the frame just recorded, so it overlaps the next tr_frame (the
 * reference presents frame n while recording frame n+1, src/main.rs:1389-1403).  `rgba8` should be pinned and must stay
 * valid until tr_wait_readback / tr_sync returns. */
TR_API int32_t tr_read_srgb8_async(tr_ctx* ctx, uint8_t* rgba8);
TR_API int32_t tr_wait_readback(tr_ctx* ctx);
TR_API int32_t tr_mip_levels(tr_ctx* ctx, uint32_t* levels);
/* per-pass device time of the last tr_frame (profiling.rs zone taxonomy). */
typedef struct {
    float cull_ms, assign_lights_ms, visibility_ms, shade_opaque_ms, allgather_ms, mips_ms,
        shade_transmission_ms, tonemap_ms, total_ms;
} tr_frame_times;
TR_API int32_t tr_enable_timing(tr_ctx* ctx, int32_t enable);
TR_API int32_t tr_read_frame_times(tr_ctx* ctx, tr_frame_times* out);
/* per-pass device time summed over the tr_frame calls since tr_enable_timing / the previous call
 * (at most the last 128 frames are kept); the reference streams the same zones to Tracy once per
 * frame (src/profiling.rs:101-131). */
TR_API int32_t tr_read_pass_totals(tr_ctx* ctx, tr_frame_times* sum, uint32_t* n_frames);

/* ------------------------------------------------------------------ */
/* glam-pbr contract batch evaluators (device arithmetic, host buffers) */
/* ------------------------------------------------------------------ */
TR_API int32_t tr_eval_basic_brdf(tr_ctx* ctx, uint32_t n, const tr_basic_brdf_params* params, tr_brdf_result* out);
TR_API int32_t tr_eval_transmission_btdf(tr_ctx* ctx, uint32_t n, const tr_transmission_btdf_params* params, tr_vec3* out);
/* the light loop of the frame kernels, one (pixel, point light) pair per element (see tr_point_light_params) */
TR_API int32_t tr_eval_point_light(tr_ctx* ctx, uint32_t n, const tr_point_light_params* params, tr_point_light_result* out);
/* samples the context's current opaque pyramid + LUT (Appendix E rules). */
TR_API int32_t tr_eval_ibl_volume_refraction(tr_ctx* ctx, uint32_t n, const tr_mat4* proj_view,
                                             const tr_ibl_volume_refraction_params* params, tr_vec3* out);

/* ------------------------------------------------------------------ */
/* Multi-GPU: one context per rank/GPU; image bands                     */
/* ------------------------------------------------------------------ */
#define TR_NCCL_UNIQUE_ID_BYTES 128
TR_API int32_t tr_comm_unique_id(uint8_t id[TR_NCCL_UNIQUE_ID_BYTES]);
TR_API int32_t tr_comm_init(tr_ctx* ctx, const uint8_t id[TR_NCCL_UNIQUE_ID_BYTES], int32_t rank, int32_t n_ranks);
TR_API int32_t tr_comm_destroy(tr_ctx* ctx);
/* Caller-balanced bands: `bounds` = n_ranks + 1 ascending row boundaries, the same on every rank (0 ... height); rank r
 * renders rows [bounds[r], bounds[r+1]).  Equal rows (tr_comm_init's default) leave the ranks unequal work where
 * coverage and light counts vary down the frame; the frame is bitwise the same for any boundaries.  Call between
 * frames, on all ranks alike. */
TR_API int32_t tr_set_bands(tr_ctx* ctx, const uint32_t* bounds, uint32_t n_bounds);
/* Peer-store path: K4 writes its band into every peer's frame directly over NVLink. */
#define TR_IPC_HANDLE_BYTES 64
TR_API int32_t tr_peer_export(tr_ctx* ctx, uint8_t handle[TR_IPC_HANDLE_BYTES]);
TR_API int32_t tr_peer_attach(tr_ctx* ctx, int32_t rank, int32_t n_ranks, const uint8_t* handles /* [n_ranks*64] */);
/* Raw device pointers, so host frameworks (torch.distributed, a Rust host) can
 * wrap the buffers without a copy.  `what` is a TR_BUF_* value. */
enum { TR_BUF_OPAQUE_MIP0 = 0, TR_BUF_HDR = 1, TR_BUF_SRGB8 = 2, TR_BUF_HDR_F32 = 3 };
TR_API int32_t tr_device_buffer(tr_ctx* ctx, int32_t what, void** device_ptr, size_t* bytes);

/* ------------------------------------------------------------------ */
/* Multi-GPU in one process: the reference's host is one thread with   */
/* one queue (src/main.rs:243, 1290-1294); a group lets that thread     */
/* drive the bands of one frame on up to 8 contexts.                    */
/* ------------------------------------------------------------------ */
/* A group joins n contexts (at most 8) of one host thread into the bands of one frame.  Member k becomes rank k of n with
 * equal-row bands; its opaque pass stores its band into every member's mip 0 through plain device pointers (peer access
 * between distinct devices, which tr_group_create enables and leaves enabled, together with access to each device's default
 * memory pool, from which tr_set_texture_async allocates), and CUDA events order the members, so no
 * call waits for the GPU inside a frame.  Contexts may share a device: 2..8 members on one GPU run exactly the code 8 GPUs
 * run.  Members must be distinct, of one size, and in no communicator (tr_comm_init), peer mapping (tr_peer_attach) or
 * other group.  While the group lives, tr_frame, tr_shade_opaque, tr_allgather_opaque, tr_set_band, tr_set_bands,
 * tr_resize, tr_comm_init, tr_peer_attach and tr_destroy on a member return TR_ERR_STATE; uploads,
 * tr_build_acceleration_structures, tr_set_stream, the timers and every tr_read_* stay per member. */
typedef struct tr_group tr_group;
/* the device set-up of src/main.rs:243 (one queue) widened to n contexts; distinct devices without peer access in both
 * directions -> TR_ERR_UNSUPPORTED */
TR_API int32_t tr_group_create(tr_ctx* const* ctxs, uint32_t n, tr_group** out_group);
/* LoopDestroyed clean-up (src/main.rs:1416-1445) of the group only: waits for every member, which then renders the whole
 * frame again as rank 0 of 1 */
TR_API int32_t tr_group_destroy(tr_group* g);
/* tr_set_bands for every member at once: n + 1 ascending row boundaries (0 ... height) */
TR_API int32_t tr_group_set_bands(tr_group* g, const uint32_t* bounds, uint32_t n_bounds);
/* swapchain-resize path (src/main.rs:996-1166) on every member; the bands return to equal rows */
TR_API int32_t tr_group_resize(tr_group* g, uint32_t width, uint32_t height);
/* one record() (src/main.rs:1551-2263) across the members: params[k] is member k's (its own
 * acceleration_structure_address when ray queries are on; normally the same camera otherwise) */
TR_API int32_t tr_group_frame(tr_group* g, const tr_frame_params* params);
/* fence wait (src/main.rs:1290) on every member */
TR_API int32_t tr_group_sync(tr_group* g);
/* the whole sRGB8 frame: every member's band into one width x height x 4 buffer */
TR_API int32_t tr_group_read_srgb8(tr_group* g, uint8_t* rgba8);
/* Copies member `source`'s scene, as its context stream sees it at the point of the call, into every other member, in
 * stream order.  addresses[k] (n entries, may be null) receives member k's acceleration-structure handle, or 0 if the
 * source has no valid top level.  Returns without waiting for the device, except where a destination buffer must grow,
 * as for the other uploads.
 * Copied: the mesh, primitives, materials, instances and lights (the buffers the source's next frame reads), uniforms,
 * the cluster AABBs of tr_build_clusters, the GGX LUT, every bound material image (with its RGBA8 levels when bound by
 * tr_set_texture_async), the culling spheres and, when the source has them, both acceleration-structure levels with their
 * refit tables; also what the source holds on the host about all of these (no read-back).  A destination then behaves as
 * a context that received the same uploads and builds: tr_update_mesh_vertices refits its trees, the top-level updates,
 * tr_set_texture_async and tr_build_acceleration_structures_async work on it.  Not copied: frame targets, G-buffers,
 * shadow masks, light lists, timers and streams.
 * Ordering: each destination's stream waits for the source stream at the call, then copies (cudaMemcpyAsync, peer to
 * peer or within one device); a frame a destination enqueued earlier reads the old scene.  The source stream then waits
 * for every destination's copies, so uploads to the source after the call do not change what the destinations receive.
 * No kernel is launched.  source >= n -> TR_ERR_INVALID_ARG; a source without a mesh -> TR_ERR_STATE; a rejected call
 * changes no member; a group of one copies nothing.  A CUDA or allocation failure part-way leaves a destination with an
 * empty scene (no mesh, no image, no structures), to be loaded again. */
TR_API int32_t tr_group_replicate_scene(tr_group* g, uint32_t source, uint64_t* addresses);

/* ------------------------------------------------------------------ */
/* Diagnostics (benchmark support; not part of the reference surface)  */
/* ------------------------------------------------------------------ */
/* kernels launched by this library in this process so far */
TR_API int32_t tr_launch_count(uint64_t* out);
/* rasteriser work since the last reset: [0] box pixels binned to tiles, [1] box pixels left after hierarchical Z,
 * [2] exact (double) coverage evaluations, [3] span pixels (fp32 depth-plane tests) */
TR_API int32_t tr_raster_stats(tr_ctx* ctx, uint64_t out[4], int32_t reset);
/* measured roofline denominators on the context's GPU: dependent-FFMA chains / STREAM-style copy */
TR_API int32_t tr_measure_fp32_peak(tr_ctx* ctx, float* tflops);
TR_API int32_t tr_measure_hbm_copy(tr_ctx* ctx, float* gbs);

#ifdef __cplusplus
}
#endif
#endif /* TR_ABI_H */
