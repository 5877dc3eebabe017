// tr_internal.h — context object and kernel launch prototypes behind include/tr_abi.h.
// The context stands in for what the reference spreads over Pipelines,
// DescriptorSets, DrawBuffers, LightBuffers and the framebuffer images
// (src/pipelines.rs, src/descriptor_sets.rs, src/main.rs:383-504, 2381-2588).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <string>
#include <vector>

#include "../../include/tr_abi.h"
#include "tr_device_accel.cuh"
#include "tr_device_pbr.cuh"

#ifndef TR_CHUNK_TRIS
#define TR_CHUNK_TRIS 64   // triangles per culling chunk of the binning pass (a multiple of 32: a warp's 32 triangles share a chunk)
#endif

namespace tr {

int32_t fail(int32_t status, const char* fmt, ...);
void count_launches(int n);  // process-wide count of kernels this library launched (tr_launch_count)
#define TR_CUDA(expr)                                                                              \
    do {                                                                                           \
        cudaError_t _e = (expr);                                                                   \
        if (_e != cudaSuccess)                                                                     \
            return tr::fail(_e == cudaErrorMemoryAllocation ? TR_ERR_OOM : TR_ERR_CUDA, "%s: %s (%s:%d)", #expr, \
                            cudaGetErrorString(_e), __FILE__, __LINE__);                           \
    } while (0)
#define TR_TRY(expr)                  \
    do {                              \
        int32_t _s = (expr);          \
        if (_s != TR_OK) return _s;   \
    } while (0)
// the frame-wide calls of a group member go through its group (tr_group.cu)
#define TR_NOT_GROUPED(c, who, instead)                                                                              \
    do {                                                                                                             \
        if ((c)->group) return tr::fail(TR_ERR_STATE, "%s: the context is a member of a group; use %s", who, instead); \
    } while (0)

struct DevBuf {
    void* p = nullptr;
    size_t bytes = 0;
    int32_t ensure(size_t n);  // grow-only
    void release();
    template <typename T> T* as() const { return reinterpret_cast<T*>(p); }
};

// The pieces of one scratch buffer: take() returns each piece's offset, 256-byte aligned, and `bytes` is what the buffer
// must hold (ensure) before the offsets are added to its base.
struct ScratchLayout {
    size_t bytes = 0;
    size_t take(size_t n) {
        const size_t o = bytes;
        bytes += (n + 255) & ~(size_t)255;
        return o;
    }
};

struct GLayer {
    DevBuf depth, normal, uv, material_id, scale, position, duv, ddepth;
    bool has_position = false;
    bool valid = false;
};

constexpr int kMaxLevels = 16;
constexpr int kMaxPeers = 8;
constexpr int kTimingRing = 128;  // frames of per-pass event pairs kept (tr_read_pass_totals)

enum Pass { P_CULL = 0, P_LIGHTS, P_VIS, P_OPAQUE, P_GATHER, P_MIPS, P_TRANS, P_TONEMAP, P_COUNT };

}  // namespace tr

struct tr_ctx {
    int device = 0;
    uint32_t width = 0, height = 0, band_y0 = 0, band_y1 = 0, flags = 0;
    cudaStream_t stream = nullptr, own_stream = nullptr;
    int sm_count = 148;

    tr::DevBuf instances, primitives, materials, lights;
    uint32_t n_instances = 0, n_primitives = 0, n_materials = 0, n_lights = 0;
    tr_uniforms uniforms{};
    bool have_uniforms = false;
    tr::DevBuf lut;
    uint32_t lut_w = 0, lut_h = 0;
    // material textures (row N2): decoded RGBA32F texels per image, descriptor table on the device.  An image bound by
    // tr_set_texture_async also holds the RGBA8 bytes of its levels behind the texels (k_textures.cu); tex_tables is the
    // device copy of texture_tables() those calls read, uploaded by the first one.
    tr::DevBuf tex_data[TR_MAX_IMAGES], tex_table, tex_tables;
    trd::TexDesc h_tex[TR_MAX_IMAGES] = {};
    bool tex_chain[TR_MAX_IMAGES] = {};   // the image's allocation holds its RGBA8 levels behind the texels (bound async)
    uint32_t n_textures = 0;          // highest bound index + 1
    bool tex_table_dirty = false;
    bool prims_alpha_clip = false;    // some primitive uses draw buffer 1 or 3 (alpha clip): the rasteriser runs the alpha test
    bool materials_textured = false;  // some material binds a texture: derivative planes + textured shading variant
    tr::DevBuf mesh_pos, mesh_nrm, mesh_uv, mesh_idx;
    uint32_t n_vertices = 0, n_indices = 0;

    // cull outputs (frustum_culling + demultiplex_draws)
    tr::DevBuf visible_ids, cull_scalars, draws[4], work_prefix, slot_z, slot_first, block_entry;
    uint32_t* d_instance_counts = nullptr;  // views into cull_scalars (state block of K1)
    uint32_t* d_cull_scalars = nullptr;     // [0] n_visible [1] visible triangles [2..5] draw_counts [6,7] ~min/max bits of slot_z
    std::vector<uint32_t> h_prim_tris, h_inst_prim;  // host copies: triangles per primitive, primitive of each instance
    // cluster culling in the binning pass (k_visibility.cu): a bounding sphere per 64 consecutive triangles of every primitive,
    // computed on the device when the mesh or the primitives change (ensure_chunks) and after every tr_update_mesh_vertices
    tr::DevBuf chunk_spheres, prim_chunk_base;   // float4 (object-space centre, radius) per chunk; first chunk of each primitive
    std::vector<uint32_t> h_chunk_base;          // the host copy of prim_chunk_base (the source of its upload)
    uint32_t n_chunks = 0;                       // spheres in chunk_spheres (0 when a primitive leaves the index buffer)
    bool chunks_valid = false, chunk_cull = false;
    std::vector<uint32_t> h_inst_mat, h_prim_first, h_prim_count;  // material of each instance; index range of each primitive
    std::vector<uint32_t> band_bounds;  // n_ranks + 1 row boundaries when the caller balances the bands itself (tr_set_bands)
    bool scene_checked = false;  // ids / index ranges validated since the last upload (validate_scene)
    uint64_t max_triangles = 0;                      // upper bound of the visibility work list
    bool tri_bound_valid = false;
    bool cull_valid = false;

    // clustered lights
    tr::DevBuf cluster_aabbs, cluster_counts, cluster_indices;
    uint32_t n_clusters = 0;
    bool clusters_valid = false, cluster_lights_valid = false;

    // frame targets
    tr::GLayer layer[2];
    tr::DevBuf vis[2], bin_entries, bin_state, tri_records, dev_status, band_list;  // sort-middle rasteriser state (k_visibility.cu)
    tr::DevBuf hdr, hdr_f32, pyramid, srgb8, mip_counter, shade_counter;
    uint32_t levels = 0, level_w[tr::kMaxLevels] = {}, level_h[tr::kMaxLevels] = {}, level_off[tr::kMaxLevels] = {};
    bool opaque_valid = false, mips_valid = false, hdr_valid = false, srgb_valid = false;

    // ray-queried shadows (k_accel.cu): bottom-level trees per primitive, top-level tree over the shadow-casting instances
    tr::DevBuf accel_tlas, accel_blas, accel_inst, accel_tris, shadow_mask[2];
    uint32_t accel_n_instances = 0;
    bool accel_blas_valid = false, accel_tlas_valid = false;
    std::vector<uint32_t> h_prim_root, h_prim_tri_base, h_prim_bucket;   // h_prim_bucket: draw_buffer_index (tr_set_primitives)
    // per-primitive table (trd::TlasPrim: object-space box, root, first triangle), uploaded by tr_build_acceleration_structures;
    // the device builder of the top level reads it (k_accel_device.cu), and so does the host one, for the boxes that a
    // bottom-level refit rewrites.  Then the device builder's scratch (grow-only).
    tr::DevBuf accel_prim_table, accel_scratch;
    // bottom-level refit after tr_update_mesh_vertices (k_mesh_update.cu): parent of every node (-1 at a root), arrival
    // counters, and the first index of every leaf-order triangle
    tr::DevBuf accel_refit;
    uint32_t accel_blas_nodes = 0, accel_n_tris = 0;
    // the scratch of the bottom level built on the device (k_accel_build.cu), grow-only
    tr::DevBuf accel_build_scratch;

    // timing (profiling.rs zone taxonomy)
    bool timing = false;
    cudaEvent_t (*ev_begin)[tr::P_COUNT] = nullptr, (*ev_end)[tr::P_COUNT] = nullptr;  // [kTimingRing][P_COUNT], lazily created
    bool (*ev_used)[tr::P_COUNT] = nullptr;
    uint64_t timing_frame = 0, timing_first = 0;  // current frame number / first frame not yet summed

    // per-frame uploads (instances, lights) from page-locked memory run ahead of the frame that uses them: on their own
    // stream, into the buffer the frame BEFORE the enqueued one read last, while the enqueued frame is still shading
    // (tr_api.cu upload_ahead).  A copy inside the compute stream costs two engine switches, ~40 us per upload.
    tr::DevBuf instances_alt, lights_alt;
    // tr_update_instance_transforms: the contiguous copy of a host source (grow-only), read by the kernel in stream order
    tr::DevBuf transform_staging;
    cudaStream_t upload_stream = nullptr;
    cudaEvent_t ev_frame_begin = nullptr, ev_inst_ready = nullptr, ev_lights_ready = nullptr;
    bool frame_begin_valid = false, inst_uploaded = false, lights_uploaded = false;   // the latter two: since the last tr_frame

    // tr_frame runs the light assignment (K2) on a side stream beside the cull and the visibility pass: they share nothing,
    // and each is a few small launches that leave most of the GPU idle
    cudaStream_t side_stream = nullptr;
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;

    // asynchronous read-back of the sRGB8 band (overlaps the next frame)
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t ev_frame_done = nullptr, ev_copy_done = nullptr;
    bool copy_pending = false;

    // multi-GPU
    int rank = 0, n_ranks = 1;
    void* nccl_comm = nullptr;
    void* peer_mip0[tr::kMaxPeers] = {};  // peer mip-0 bases (self included) for the peer-store path
    uint32_t* peer_flags[tr::kMaxPeers] = {};  // every rank's barrier words (self included), behind its pyramid
    size_t barrier_flags_offset = 0;      // byte offset of the barrier words inside the pyramid allocation
    uint32_t barrier_epoch = 0;
    bool peers_attached = false;
    tr_group* group = nullptr;            // single-process group this context is rank `rank` of (tr_group.cu)
};

// tr_group_create: contexts of one host thread joined into the bands of one frame.  Member k is rank k; its opaque pass
// stores into every member's mip 0 through plain device pointers, and CUDA events order the members (tr_group.cu).
struct tr_group {
    int n = 0;
    tr_ctx* members[tr::kMaxPeers] = {};
    cudaEvent_t ev_front[tr::kMaxPeers] = {};  // recorded after member k's opaque pass (its band is in every mip 0)
    cudaEvent_t ev_back[tr::kMaxPeers] = {};   // recorded after member k's transmissive pass (done reading its mip 0)
    // tr_group_replicate_scene: on the source, the point of the call; on a destination, the end of its copies
    cudaEvent_t ev_replica[tr::kMaxPeers] = {};
};

namespace tr {

// ---- kernel launchers (each in its own .cu) ---------------------------------
struct ShadeLaunch {
    uint32_t width, height, px_begin, px_end;
    const float* depth;
    const float* normal;
    const uint32_t* material_id;
    const float* scale;     // transmissive layer
    const float* position;  // optional
    const float* uv;        // textured materials only
    const float4* duv;
    const float2* ddepth;
    const trd::TexDesc* textures;  // nullptr: no material binds a texture
    uint32_t n_textures;
    const tr_material_info* materials;
    const tr_light* lights;
    uint32_t n_lights;
    const uint32_t* cluster_counts;
    const uint32_t* cluster_indices;
    uint32_t n_clusters;
    tr_uniforms uniforms;
    trd::mat4 proj_view, inv_proj_view;
    float view_position[3];
    uint32_t framebuffer_size_x;
    float log2_size_x;
    uint2* hdr;                    // RGBA16F
    float4* hdr_f32;               // optional
    uint2* opaque[kMaxPeers];      // sampled opaque mip 0 on this GPU [0] and, for the peer-store path, on every peer
    int n_opaque;
    trd::PyramidDesc pyramid;
    trd::LutDesc lut;
    // ray-queried shadows: occluded-ray bits per pixel, written by the shadow pass and read by the shading kernel.
    // Five planes of `shadow_plane` words: 0-3 = position in the cluster's light list, 4 = the sun.  nullptr: no ray queries.
    uint32_t* chunk_counter;  // work counter of the shading kernels (zeroed before every launch)
    uint32_t* shadow_mask;
    uint32_t shadow_plane;
    trd::AccelDesc accel;
};

int32_t launch_shade_opaque(const ShadeLaunch& p, int sm_count, cudaStream_t s);
int32_t launch_shade_transmission(const ShadeLaunch& p, int sm_count, cudaStream_t s);
// the same kernels instantiated with the shadow-mask reads, plus the pass that traces the rays (k_shade_shadow.cu)
int32_t launch_shade_opaque_shadowed(const ShadeLaunch& p, int sm_count, cudaStream_t s);
int32_t launch_shade_transmission_shadowed(const ShadeLaunch& p, int sm_count, cudaStream_t s);
int32_t launch_shadow_mask(const ShadeLaunch& p, int sm_count, cudaStream_t s);
trd::AccelDesc accel_desc(const tr_ctx* c);
int32_t accel_build(tr_ctx* c);       // bottom-level structures of every primitive, then the top level
int32_t accel_build_tlas(tr_ctx* c);  // top level only (instances moved)
// the top level built on the device in stream order (k_accel_device.cu); launches kAsyncTlasLaunches kernels
int32_t accel_build_tlas_async(tr_ctx* c);
constexpr int kAsyncTlasLaunches = 19;
// the bottom level built on the device in stream order, then the top level (k_accel_build.cu); launches
// async_blas_launches(n_primitives) + kAsyncTlasLaunches kernels
int32_t accel_build_async(tr_ctx* c);
int async_blas_launches(uint32_t n_primitives);
void launch_block_scan(uint32_t* data, uint32_t len, cudaStream_t s);   // exclusive, one block (k_accel_device.cu)
// tr_update_mesh_vertices (k_mesh_update.cu): the chunk spheres in one launch, the bottom-level refit in two
int32_t launch_chunk_spheres(tr_ctx* c);
int32_t accel_refit_blas(tr_ctx* c);
constexpr int kChunkSphereLaunches = 1;
constexpr int kRefitLaunches = 2;
// tr_update_instance_transforms (k_instances.cu): the n similarities at `src` (device memory) into the transforms of
// instances [first, first + n), ids kept; one launch
int32_t launch_instance_transforms(tr_ctx* c, uint32_t first, uint32_t n, const tr_packed_similarity* src);
constexpr int kInstanceTransformLaunches = 1;
// The decode and encode tables of the material images (k_textures.cu), built once on the host: the float tables of the
// store, which tr_set_texture uses too, and the float64 decode tables and sRGB encode thresholds of the device mip chain.
struct TexTables {
    double dec64[2][256];   // [0] sRGB colour -> linear, [1] v / 255.0 (alpha, UNORM)
    double encode[256];     // encode[k - 1]: the least x whose sRGB byte is >= k; encode[255] = 2.0
    float dec32[2][256];    // the store's texels: (float) of dec64[0], and (float)v / 255.0f
};
const TexTables& texture_tables();
// tr_set_texture_async: level 0 from the bytes at `chain` (already in stream order) into d.base, then levels 1 .. d.levels - 1
// (bytes and texels); d.levels launches
int32_t launch_texture_chain(const TexTables* d_tables, const trd::TexDesc& d, uint8_t* chain, int sm_count, cudaStream_t s);
int32_t launch_trace_rays(tr_ctx* c, uint32_t n, const float* d_origins, const float* d_directions, const float* d_t_max, uint8_t* d_lit);
int32_t launch_generate_mips(uint2* pyramid, uint32_t levels, const uint32_t* w, const uint32_t* h, const uint32_t* off,
                             uint32_t* counter, int sm_count, cudaStream_t s);
int32_t launch_tonemap(const uint2* hdr, uchar4* out, uint32_t px_begin, uint32_t px_end,
                       const tr_baked_lottes_tonemapper_params& params, int sm_count, cudaStream_t s);
int32_t launch_cull(tr_ctx* c, const tr_culling_push_constants& pc);
int32_t launch_build_clusters(tr_ctx* c, const tr_write_cluster_data_push_constants& pc);
int32_t launch_assign_lights(tr_ctx* c, const tr_assign_lights_push_constants& pc);
int32_t launch_visibility(tr_ctx* c, const tr_push_constants& pc);
int32_t launch_eval_basic_brdf(uint32_t n, const tr_basic_brdf_params* in, tr_brdf_result* out, cudaStream_t s);
int32_t launch_eval_transmission_btdf(uint32_t n, const tr_transmission_btdf_params* in, tr_vec3* out, cudaStream_t s);
int32_t launch_eval_point_light(uint32_t n, const tr_point_light_params* in, tr_point_light_result* out, cudaStream_t s);
int32_t launch_eval_ibl(uint32_t n, const trd::mat4& pv, const tr_ibl_volume_refraction_params* in, tr_vec3* out,
                        const trd::PyramidDesc& pyr, const trd::LutDesc& lut, cudaStream_t s);

int32_t check_device_status(tr_ctx* c, const char* who);
int32_t ensure_tri_bound(tr_ctx* c, const char* who);   // max_triangles: the work list's upper bound
int32_t ensure_chunks(tr_ctx* c);   // (re)builds chunk_spheres / prim_chunk_base after a mesh or primitive upload, in stream order
int32_t validate_scene(tr_ctx* c, const char* who);  // instance -> primitive / material ids, primitive index ranges  // sticky device-side error bits -> TR_ERR_STATE
void mat4_inverse_f64(const tr_mat4& m, tr_mat4* out);
int32_t ensure_layer(tr_ctx* c, int layer, bool with_position);
int32_t upload_texture_table(tr_ctx* c);  // descriptor table of the bound images -> device (if it changed)
// tr_group_replicate_scene (tr_group.cu): src's scene into dst on dst's stream, which must already wait for the point of the
// call on src's stream; copies only, no kernel
int32_t replicate_scene(tr_ctx* dst, const tr_ctx* src);
void band_of(const tr_ctx* c, int r, uint32_t* y0, uint32_t* y1);   // rows of rank r (tr_comm.cu)

// tr_frame in pieces (tr_api.cu), shared with tr_group_frame (tr_group.cu):
//   frame_front   per-pass timer mark, ev_frame_begin, K2 on the side stream beside K1 + K3, join
//   shade_opaque  K4 (tr_shade_opaque without the group check); a group member stores its band into every member's mip 0
//   frame_back    K5, K6, then records `after_transmission` (if not null) on the context stream, then K7
int32_t frame_front(tr_ctx* c, const tr_frame_params* f);
int32_t shade_opaque(tr_ctx* c, const tr_push_constants* pc);
int32_t frame_back(tr_ctx* c, const tr_frame_params* f, cudaEvent_t after_transmission);
int32_t check_pc(const tr_ctx* c, const tr_push_constants* pc, const char* who);
int32_t resize_frame(tr_ctx* c, uint32_t width, uint32_t height);   // tr_resize after its checks
void pass_begin(tr_ctx* c, int pass);
void pass_end(tr_ctx* c, int pass);

}  // namespace tr
