// tr_api.cu — the extern "C" boundary (include/tr_abi.h): context lifecycle, uploads,
// per-frame pass entry points in record() order (src/main.rs:1551-2263) and parity hooks.
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <atomic>
#include <new>
#include <vector>

#include <algorithm>

#include "tr_internal.h"

namespace tr {

static thread_local char g_err[512] = "";
static std::atomic<uint64_t> g_launches{0};
void count_launches(int n) { g_launches.fetch_add((uint64_t)n, std::memory_order_relaxed); }

int32_t fail(int32_t status, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return status;
}

int32_t DevBuf::ensure(size_t n) {
    if (n == 0) n = 16;
    if (n <= bytes) return TR_OK;
    if (p) cudaFree(p);
    p = nullptr;
    bytes = 0;
    cudaError_t e = cudaMalloc(&p, n);
    if (e != cudaSuccess) {
        p = nullptr;
        return fail(e == cudaErrorMemoryAllocation ? TR_ERR_OOM : TR_ERR_CUDA, "cudaMalloc(%zu): %s", n,
                    cudaGetErrorString(e));
    }
    bytes = n;
    return TR_OK;
}

void DevBuf::release() {
    if (p && bytes) cudaFree(p);
    p = nullptr;
    bytes = 0;
}

// inverse(proj_view) for the G-buffer position decode: cofactor expansion in double, rounded to
// f32 once (same rule as the oracle's orc_mat4_inverse).
void mat4_inverse_f64(const tr_mat4& m, tr_mat4* out) {
    const float* f = reinterpret_cast<const float*>(&m);
    double a[16], v[16];
    for (int i = 0; i < 16; i++) a[i] = (double)f[i];
    v[0] = a[5] * a[10] * a[15] - a[5] * a[11] * a[14] - a[9] * a[6] * a[15] + a[9] * a[7] * a[14] + a[13] * a[6] * a[11] - a[13] * a[7] * a[10];
    v[4] = -a[4] * a[10] * a[15] + a[4] * a[11] * a[14] + a[8] * a[6] * a[15] - a[8] * a[7] * a[14] - a[12] * a[6] * a[11] + a[12] * a[7] * a[10];
    v[8] = a[4] * a[9] * a[15] - a[4] * a[11] * a[13] - a[8] * a[5] * a[15] + a[8] * a[7] * a[13] + a[12] * a[5] * a[11] - a[12] * a[7] * a[9];
    v[12] = -a[4] * a[9] * a[14] + a[4] * a[10] * a[13] + a[8] * a[5] * a[14] - a[8] * a[6] * a[13] - a[12] * a[5] * a[10] + a[12] * a[6] * a[9];
    v[1] = -a[1] * a[10] * a[15] + a[1] * a[11] * a[14] + a[9] * a[2] * a[15] - a[9] * a[3] * a[14] - a[13] * a[2] * a[11] + a[13] * a[3] * a[10];
    v[5] = a[0] * a[10] * a[15] - a[0] * a[11] * a[14] - a[8] * a[2] * a[15] + a[8] * a[3] * a[14] + a[12] * a[2] * a[11] - a[12] * a[3] * a[10];
    v[9] = -a[0] * a[9] * a[15] + a[0] * a[11] * a[13] + a[8] * a[1] * a[15] - a[8] * a[3] * a[13] - a[12] * a[1] * a[11] + a[12] * a[3] * a[9];
    v[13] = a[0] * a[9] * a[14] - a[0] * a[10] * a[13] - a[8] * a[1] * a[14] + a[8] * a[2] * a[13] + a[12] * a[1] * a[10] - a[12] * a[2] * a[9];
    v[2] = a[1] * a[6] * a[15] - a[1] * a[7] * a[14] - a[5] * a[2] * a[15] + a[5] * a[3] * a[14] + a[13] * a[2] * a[7] - a[13] * a[3] * a[6];
    v[6] = -a[0] * a[6] * a[15] + a[0] * a[7] * a[14] + a[4] * a[2] * a[15] - a[4] * a[3] * a[14] - a[12] * a[2] * a[7] + a[12] * a[3] * a[6];
    v[10] = a[0] * a[5] * a[15] - a[0] * a[7] * a[13] - a[4] * a[1] * a[15] + a[4] * a[3] * a[13] + a[12] * a[1] * a[7] - a[12] * a[3] * a[5];
    v[14] = -a[0] * a[5] * a[14] + a[0] * a[6] * a[13] + a[4] * a[1] * a[14] - a[4] * a[2] * a[13] - a[12] * a[1] * a[6] + a[12] * a[2] * a[5];
    v[3] = -a[1] * a[6] * a[11] + a[1] * a[7] * a[10] + a[5] * a[2] * a[11] - a[5] * a[3] * a[10] - a[9] * a[2] * a[7] + a[9] * a[3] * a[6];
    v[7] = a[0] * a[6] * a[11] - a[0] * a[7] * a[10] - a[4] * a[2] * a[11] + a[4] * a[3] * a[10] + a[8] * a[2] * a[7] - a[8] * a[3] * a[6];
    v[11] = -a[0] * a[5] * a[11] + a[0] * a[7] * a[9] + a[4] * a[1] * a[11] - a[4] * a[3] * a[9] - a[8] * a[1] * a[7] + a[8] * a[3] * a[5];
    v[15] = a[0] * a[5] * a[10] - a[0] * a[6] * a[9] - a[4] * a[1] * a[10] + a[4] * a[2] * a[9] + a[8] * a[1] * a[6] - a[8] * a[2] * a[5];
    const double det = a[0] * v[0] + a[1] * v[4] + a[2] * v[8] + a[3] * v[12];
    const double r = 1.0 / det;
    float* o = reinterpret_cast<float*>(out);
    for (int i = 0; i < 16; i++) o[i] = (float)(v[i] * r);
}

static uint32_t mip_levels_for_size(uint32_t w, uint32_t h) {  // src/main.rs:2590-2592
    const uint32_t m = w < h ? w : h;
    return (uint32_t)log2f((float)m) + 1u;
}

static int32_t alloc_frame(tr_ctx* c) {
    const size_t npx = (size_t)c->width * c->height;
    c->levels = mip_levels_for_size(c->width, c->height);
    if (c->levels > (uint32_t)kMaxLevels) return fail(TR_ERR_INVALID_ARG, "too many mip levels");
    uint32_t w = c->width, h = c->height, off = 0;
    for (uint32_t l = 0; l < c->levels; l++) {
        c->level_w[l] = w;
        c->level_h[l] = h;
        c->level_off[l] = off;
        off += ((w * h + 1u) & ~1u);  // keep every level 16-byte aligned
        w = w / 2 > 1 ? w / 2 : 1;
        h = h / 2 > 1 ? h / 2 : 1;
    }
    c->barrier_flags_offset = (size_t)off * 8;  // 256 bytes of cross-GPU barrier words live behind the last mip level
    TR_TRY(c->pyramid.ensure((size_t)off * 8 + 256));
    TR_TRY(c->hdr.ensure(npx * 8));
    TR_TRY(c->srgb8.ensure(npx * 4));
    if (c->flags & TR_FLAG_HDR_F32_DEBUG) TR_TRY(c->hdr_f32.ensure(npx * 16));
    TR_TRY(c->mip_counter.ensure(16));
    TR_CUDA(cudaMemsetAsync(c->mip_counter.p, 0, 16, c->stream));
    for (int l = 0; l < 2; l++) c->layer[l].valid = false;
    c->opaque_valid = c->mips_valid = c->hdr_valid = c->srgb_valid = false;
    return TR_OK;
}

int32_t ensure_layer(tr_ctx* c, int layer, bool with_position) {
    const size_t npx = (size_t)c->width * c->height;
    GLayer& g = c->layer[layer];
    TR_TRY(g.depth.ensure(npx * 4));
    TR_TRY(g.normal.ensure(npx * 12));
    TR_TRY(g.uv.ensure(npx * 8));
    TR_TRY(g.material_id.ensure(npx * 4));
    TR_TRY(g.scale.ensure(npx * 4));
    if (with_position) TR_TRY(g.position.ensure(npx * 12));
    if (c->materials_textured) {  // derivative planes exist only while some material binds a texture
        const bool fresh = g.duv.bytes < npx * 16;
        TR_TRY(g.duv.ensure(npx * 16));
        TR_TRY(g.ddepth.ensure(npx * 8));
        if (fresh) {
            TR_CUDA(cudaMemsetAsync(g.duv.p, 0, npx * 16, c->stream));
            TR_CUDA(cudaMemsetAsync(g.ddepth.p, 0, npx * 8, c->stream));
        }
    }
    return TR_OK;
}

int32_t upload_texture_table(tr_ctx* c) {
    if (c->tex_table_dirty || !c->tex_table.p) {
        TR_TRY(c->tex_table.ensure(sizeof(trd::TexDesc) * TR_MAX_IMAGES));
        TR_CUDA(cudaMemcpyAsync(c->tex_table.p, c->h_tex, sizeof(trd::TexDesc) * TR_MAX_IMAGES, cudaMemcpyHostToDevice, c->stream));
        c->tex_table_dirty = false;
    }
    return TR_OK;
}

static trd::PyramidDesc pyramid_desc(const tr_ctx* c) {
    trd::PyramidDesc d{};
    d.base = c->pyramid.as<uint2>();
    d.levels = c->levels;
    for (uint32_t l = 0; l < c->levels; l++) {
        d.w[l] = c->level_w[l];
        d.h[l] = c->level_h[l];
        d.offset[l] = c->level_off[l];
    }
    return d;
}

static trd::LutDesc lut_desc(const tr_ctx* c) {
    trd::LutDesc d{};
    d.rg = c->lut.as<uchar2>();
    d.w = c->lut_w;
    d.h = c->lut_h;
    return d;
}

static int slot_of(const tr_ctx* c) { return (int)(c->timing_frame % kTimingRing); }
void pass_begin(tr_ctx* c, int pass) {
    if (!c->timing) return;
    const int slot = (int)(c->timing_frame % kTimingRing);
    cudaEventRecord(c->ev_begin[slot][pass], c->stream);
    c->ev_used[slot][pass] = true;
}
void pass_end(tr_ctx* c, int pass) {
    if (!c->timing) return;
    cudaEventRecord(c->ev_end[slot_of(c)][pass], c->stream);
}
static void timing_next_frame(tr_ctx* c) {
    if (!c->timing) return;
    c->timing_frame++;
    if (c->timing_frame - c->timing_first >= (uint64_t)kTimingRing) c->timing_first = c->timing_frame - kTimingRing + 1;
    const int slot = slot_of(c);
    for (int i = 0; i < P_COUNT; i++) c->ev_used[slot][i] = false;
}
static int32_t sum_frame_times(tr_ctx* c, int slot, tr_frame_times* out) {
    float* dst[P_COUNT] = {&out->cull_ms, &out->assign_lights_ms, &out->visibility_ms, &out->shade_opaque_ms,
                           &out->allgather_ms, &out->mips_ms, &out->shade_transmission_ms, &out->tonemap_ms};
    int first = -1, last = -1;
    for (int i = 0; i < P_COUNT; i++) {
        if (!c->ev_used[slot][i]) continue;
        float ms = 0.0f;
        if (cudaEventElapsedTime(&ms, c->ev_begin[slot][i], c->ev_end[slot][i]) == cudaSuccess) *dst[i] += ms;
        if (first < 0) first = i;
        last = i;
    }
    if (first >= 0) {
        float ms = 0.0f;
        if (cudaEventElapsedTime(&ms, c->ev_begin[slot][first], c->ev_end[slot][last]) == cudaSuccess) out->total_ms += ms;
    }
    return first >= 0 ? 1 : 0;
}

int32_t check_pc(const tr_ctx* c, const tr_push_constants* pc, const char* who) {
    if (!pc) return fail(TR_ERR_INVALID_ARG, "%s: null push constants", who);
    if (pc->acceleration_structure_address != 0) {  // the `--ray-tracing` variant of the fragment shaders, lib.rs:100-102
        if (!c->accel_blas_valid || pc->acceleration_structure_address != (uint64_t)(uintptr_t)c->accel_tlas.p)
            return fail(TR_ERR_INVALID_ARG, "%s: acceleration_structure_address is not the handle of tr_build_acceleration_structures "
                        "(or the mesh / primitives changed since)", who);
        if (!c->accel_tlas_valid)
            return fail(TR_ERR_STATE, "%s: instances or mesh vertices changed since the top-level structure was built "
                        "(tr_update_top_level_acceleration_structure)", who);
    }
    if (pc->framebuffer_size.x != c->width || pc->framebuffer_size.y != c->height)
        return fail(TR_ERR_INVALID_ARG, "%s: framebuffer_size %ux%u does not match the context %ux%u", who,
                    pc->framebuffer_size.x, pc->framebuffer_size.y, c->width, c->height);
    return TR_OK;
}

static int32_t ensure_cluster_lists(tr_ctx* c, const char* who) {
    if (c->cluster_lights_valid) return TR_OK;
    if (c->n_lights != 0) return fail(TR_ERR_STATE, "%s: light lists missing (tr_assign_lights / tr_set_cluster_lights)", who);
    TR_TRY(c->cluster_counts.ensure((size_t)c->n_clusters * 4));
    TR_TRY(c->cluster_indices.ensure((size_t)c->n_clusters * TR_MAX_LIGHTS_PER_CLUSTER * 4));
    TR_CUDA(cudaMemsetAsync(c->cluster_counts.p, 0, (size_t)c->n_clusters * 4, c->stream));
    c->cluster_lights_valid = true;
    return TR_OK;
}

static int32_t fill_shade(tr_ctx* c, const tr_push_constants* pc, int layer, ShadeLaunch* s, const char* who) {
    TR_TRY(check_pc(c, pc, who));
    if (!c->have_uniforms) return fail(TR_ERR_STATE, "%s: uniforms not set", who);
    if (!c->n_materials) return fail(TR_ERR_STATE, "%s: materials not set", who);
    if (!c->layer[layer].valid) return fail(TR_ERR_STATE, "%s: no G-buffer for layer %d (tr_visibility / tr_set_gbuffer)", who, layer);
    TR_TRY(validate_scene(c, who));
    TR_TRY(ensure_cluster_lists(c, who));
    const GLayer& g = c->layer[layer];
    memset(s, 0, sizeof(*s));
    s->width = c->width;
    s->height = c->height;
    s->px_begin = c->band_y0 * c->width;
    s->px_end = c->band_y1 * c->width;
    s->depth = g.depth.as<float>();
    s->normal = g.normal.as<float>();
    s->material_id = g.material_id.as<uint32_t>();
    s->scale = g.scale.as<float>();
    s->position = g.has_position ? g.position.as<float>() : nullptr;
    if (c->materials_textured) {
        TR_TRY(ensure_layer(c, layer, g.has_position));
        TR_TRY(upload_texture_table(c));
        s->uv = g.uv.as<float>();
        s->duv = g.duv.as<float4>();
        s->ddepth = g.ddepth.as<float2>();
        s->textures = c->tex_table.as<trd::TexDesc>();
        s->n_textures = c->n_textures;
    }
    s->materials = c->materials.as<tr_material_info>();
    s->lights = c->lights.as<tr_light>();
    s->n_lights = c->n_lights;
    s->cluster_counts = c->cluster_counts.as<uint32_t>();
    s->cluster_indices = c->cluster_indices.as<uint32_t>();
    s->n_clusters = c->n_clusters;
    s->uniforms = c->uniforms;
    memcpy(&s->proj_view, &pc->proj_view, sizeof(trd::mat4));
    tr_mat4 inv;
    mat4_inverse_f64(pc->proj_view, &inv);
    memcpy(&s->inv_proj_view, &inv, sizeof(trd::mat4));
    s->view_position[0] = pc->view_position.x;
    s->view_position[1] = pc->view_position.y;
    s->view_position[2] = pc->view_position.z;
    s->framebuffer_size_x = pc->framebuffer_size.x;
    s->log2_size_x = log2f((float)pc->framebuffer_size.x);  // glam-pbr lib.rs:334-335, per-frame constant
    s->hdr = c->hdr.as<uint2>();
    s->hdr_f32 = (c->flags & TR_FLAG_HDR_F32_DEBUG) ? c->hdr_f32.as<float4>() : nullptr;
    s->pyramid = pyramid_desc(c);
    s->lut = lut_desc(c);
    TR_TRY(c->shade_counter.ensure(256));
    s->chunk_counter = c->shade_counter.as<uint32_t>();
    if (pc->acceleration_structure_address != 0) {
        const size_t plane = (size_t)c->width * c->height;
        TR_TRY(c->shadow_mask[layer].ensure(plane * 5 * 4));
        s->shadow_mask = c->shadow_mask[layer].as<uint32_t>();
        s->shadow_plane = (uint32_t)plane;
        s->accel = accel_desc(c);
    }
    return TR_OK;
}

// The kernels index primitives[instance.primitive_id], materials[instance.material_id] and the index buffer at
// first_index .. first_index + index_count without bounds checks of their own (neither do the reference's shaders —
// shader/src/lib.rs:393-399 `index_unchecked`); the ids are checked here, once per upload, on the host copies.
int32_t validate_scene(tr_ctx* c, const char* who) {
    if (c->scene_checked) return TR_OK;
    for (uint32_t i = 0; i < c->n_instances; i++) {
        if (c->h_inst_prim[i] >= c->n_primitives)
            return fail(TR_ERR_INVALID_ARG, "%s: instance %u names primitive %u of %u", who, i, c->h_inst_prim[i], c->n_primitives);
        if (c->n_materials && c->h_inst_mat[i] >= c->n_materials)
            return fail(TR_ERR_INVALID_ARG, "%s: instance %u names material %u of %u", who, i, c->h_inst_mat[i], c->n_materials);
    }
    if (c->n_indices)
        for (uint32_t p = 0; p < c->n_primitives; p++)
            if ((uint64_t)c->h_prim_first[p] + c->h_prim_count[p] > c->n_indices)
                return fail(TR_ERR_INVALID_ARG, "%s: primitive %u reads indices [%u, %u + %u) of %u", who, p, c->h_prim_first[p],
                            c->h_prim_first[p], c->h_prim_count[p], c->n_indices);
    c->scene_checked = true;
    return TR_OK;
}

// A bounding sphere (object space) per TR_CHUNK_TRIS consecutive triangles of every primitive: the binning pass tests it
// against the frustum and the band before it touches the chunk's vertices.  Centre = centre of the chunk's box, radius = the
// farthest vertex (double, rounded up); computed on the device in stream order (k_mesh_update.cu), so tr_update_mesh_vertices
// can redo it every frame.  Without a mesh, or with a primitive that leaves the index buffer, the test is off.
int32_t ensure_chunks(tr_ctx* c) {
    if (c->chunks_valid) return TR_OK;
    std::vector<uint32_t>& base = c->h_chunk_base;   // kept: the source of an upload that does not wait
    base.assign((size_t)c->n_primitives + 1, 0u);
    uint32_t n = 0;
    bool ok = c->n_indices != 0;
    for (uint32_t p = 0; ok && p < c->n_primitives; p++) {
        const uint64_t first = c->h_prim_first[p], tris = c->h_prim_count[p] / 3;
        if (first + tris * 3 > c->n_indices) { ok = false; break; }   // validate_scene reports it
        base[p] = n;
        n += (uint32_t)((tris + TR_CHUNK_TRIS - 1) / TR_CHUNK_TRIS);
    }
    base[c->n_primitives] = n;
    TR_TRY(c->prim_chunk_base.ensure(base.size() * 4));
    TR_TRY(c->chunk_spheres.ensure(std::max<size_t>((size_t)n * 16, 16)));
    TR_CUDA(cudaMemcpyAsync(c->prim_chunk_base.p, base.data(), base.size() * 4, cudaMemcpyHostToDevice, c->stream));
    c->n_chunks = ok ? n : 0u;
    c->chunk_cull = ok && !getenv("TR_NO_CHUNK_CULL");
    c->chunks_valid = true;
    return launch_chunk_spheres(c);
}

// Upper bound of the visibility work list (every instance visible), recomputed after an instance / primitive upload.
int32_t ensure_tri_bound(tr_ctx* c, const char* who) {
    if (c->tri_bound_valid) return TR_OK;
    uint64_t n = 0;
    for (uint32_t pid : c->h_inst_prim) {
        if (pid >= c->h_prim_tris.size()) return fail(TR_ERR_INVALID_ARG, "%s: an instance names primitive %u of %zu", who, pid, c->h_prim_tris.size());
        n += c->h_prim_tris[pid];
    }
    if (n >= (1ull << 31)) return fail(TR_ERR_UNSUPPORTED, "%s: more than 2^31 triangles", who);
    c->max_triangles = n;
    c->tri_bound_valid = true;
    return TR_OK;
}

int32_t check_device_status(tr_ctx* c, const char* who) {
    if (!c->dev_status.p) return TR_OK;
    uint32_t bits = 0;
    TR_CUDA(cudaMemcpyAsync(&bits, c->dev_status.p, 4, cudaMemcpyDeviceToHost, c->stream));
    TR_CUDA(cudaStreamSynchronize(c->stream));
    if (bits == 0) return TR_OK;
    cudaMemsetAsync(c->dev_status.p, 0, 4, c->stream);
    return fail(TR_ERR_STATE, "%s: the visibility pass overflowed its work lists (bits %u: 1 = triangle records, 2 = tile bins); "
                              "the G-buffer of that frame is incomplete", who, bits);
}

int32_t resize_frame(tr_ctx* c, uint32_t width, uint32_t height) {
    c->width = width;
    c->height = height;
    c->band_y0 = 0;
    c->band_y1 = height;
    c->band_bounds.clear();
    if (c->n_ranks > 1) {  // a rank of a band-sharded frame keeps its (equal-rows) share of the new frame
        c->band_y0 = (uint32_t)(((uint64_t)c->rank * height) / c->n_ranks);
        c->band_y1 = (uint32_t)(((uint64_t)(c->rank + 1) * height) / c->n_ranks);
    }
    c->clusters_valid = false;  // main.rs:1113-1121 reruns write_cluster_data on resize
    return alloc_frame(c);
}

// ------------------------------------------------------------------ tr_frame in pieces (tr_internal.h)
int32_t frame_front(tr_ctx* c, const tr_frame_params* f) {
    timing_next_frame(c);
    // everything the previous frame read is free from here on: the mark the next frame's uploads wait for (upload_ahead)
    if (!c->ev_frame_begin) TR_CUDA(cudaEventCreateWithFlags(&c->ev_frame_begin, cudaEventDisableTiming));
    TR_CUDA(cudaEventRecord(c->ev_frame_begin, c->stream));
    c->frame_begin_valid = true;
    c->inst_uploaded = c->lights_uploaded = false;
    const bool side = c->n_lights && !(f->flags & TR_FRAME_SKIP_VISIBILITY);
    if (side) {   // K2 beside K1 + K3: fork here, join before the opaque pass reads the light lists
        if (!c->side_stream) {
            TR_CUDA(cudaStreamCreateWithFlags(&c->side_stream, cudaStreamNonBlocking));
            TR_CUDA(cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming));
            TR_CUDA(cudaEventCreateWithFlags(&c->ev_join, cudaEventDisableTiming));
        }
        TR_CUDA(cudaEventRecord(c->ev_fork, c->stream));
        TR_CUDA(cudaStreamWaitEvent(c->side_stream, c->ev_fork, 0));
        cudaStream_t main_stream = c->stream;
        c->stream = c->side_stream;            // the pass and its timer events go to the side stream
        const int32_t st = tr_assign_lights(c, &f->assign_lights);
        c->stream = main_stream;
        if (st != TR_OK) return st;
        TR_CUDA(cudaEventRecord(c->ev_join, c->side_stream));
    } else if (c->n_lights) {
        TR_TRY(tr_assign_lights(c, &f->assign_lights));
    }
    if (!(f->flags & TR_FRAME_SKIP_VISIBILITY)) {
        TR_TRY(tr_cull(c, &f->culling));
        TR_TRY(tr_visibility(c, &f->push_constants));
    }
    if (side) TR_CUDA(cudaStreamWaitEvent(c->stream, c->ev_join, 0));
    return TR_OK;
}

int32_t shade_opaque(tr_ctx* c, const tr_push_constants* pc) {
    ShadeLaunch s;
    TR_TRY(fill_shade(c, pc, TR_LAYER_OPAQUE, &s, "tr_shade_opaque"));
    uint2* mip0 = c->pyramid.as<uint2>() + c->level_off[0];
    s.n_opaque = 0;
    if (c->group) {   // every member's mip 0, this one's included: plain device pointers (same device or peer access)
        for (int r = 0; r < c->group->n; r++) {
            const tr_ctx* m = c->group->members[r];
            s.opaque[s.n_opaque++] = m->pyramid.as<uint2>() + m->level_off[0];
        }
    } else if (c->peers_attached) {
        for (int r = 0; r < c->n_ranks; r++) s.opaque[s.n_opaque++] = reinterpret_cast<uint2*>(c->peer_mip0[r]);
    } else {
        s.opaque[s.n_opaque++] = mip0;
    }
    pass_begin(c, P_OPAQUE);
    if (s.shadow_mask) {
        TR_TRY(launch_shadow_mask(s, c->sm_count, c->stream));
        TR_TRY(launch_shade_opaque_shadowed(s, c->sm_count, c->stream));
    } else {
        TR_TRY(launch_shade_opaque(s, c->sm_count, c->stream));
    }
    pass_end(c, P_OPAQUE);
    c->opaque_valid = true;
    c->hdr_valid = true;
    c->mips_valid = false;
    return TR_OK;
}

int32_t frame_back(tr_ctx* c, const tr_frame_params* f, cudaEvent_t after_transmission) {
    TR_TRY(tr_generate_mips(c));
    if (c->layer[TR_LAYER_TRANSMISSIVE].valid) TR_TRY(tr_shade_transmission(c, &f->push_constants));
    if (after_transmission) TR_CUDA(cudaEventRecord(after_transmission, c->stream));
    if (!(f->flags & TR_FRAME_SKIP_TONEMAP)) TR_TRY(tr_tonemap(c, &f->tonemap));
    return TR_OK;
}

int32_t comm_allgather_opaque(tr_ctx* c);  // tr_comm.cu
int32_t comm_barrier(tr_ctx* c);
void comm_release(tr_ctx* c);

}  // namespace tr

using namespace tr;

#define TR_CHECK_CTX(c)                                                     \
    do {                                                                    \
        if (!(c)) return tr::fail(TR_ERR_INVALID_ARG, "null context");      \
        cudaError_t _e = cudaSetDevice((c)->device);                        \
        if (_e != cudaSuccess) return tr::fail(TR_ERR_CUDA, "cudaSetDevice(%d): %s", (c)->device, cudaGetErrorString(_e)); \
    } while (0)

extern "C" {

const char* tr_last_error(void) { return tr::g_err; }
const char* tr_version(void) { return "transmission_renderer_b200 0.1 (sm_100a)"; }

int32_t tr_create(const tr_config* config, tr_ctx** out_ctx) {
    if (!config || !out_ctx) return fail(TR_ERR_INVALID_ARG, "tr_create: null argument");
    *out_ctx = nullptr;
    if (config->width == 0 || config->height == 0) return fail(TR_ERR_INVALID_ARG, "tr_create: empty framebuffer");
    int n_dev = 0;
    cudaError_t e = cudaGetDeviceCount(&n_dev);
    if (e != cudaSuccess || n_dev == 0)
        return fail(TR_ERR_CUDA, "tr_create: no CUDA device (%s); this library has no CPU path",
                    e != cudaSuccess ? cudaGetErrorString(e) : "device count 0");
    if (config->device < 0 || config->device >= n_dev) return fail(TR_ERR_INVALID_ARG, "tr_create: device %d of %d", config->device, n_dev);
    TR_CUDA(cudaSetDevice(config->device));
    tr_ctx* c = new (std::nothrow) tr_ctx();
    if (!c) return fail(TR_ERR_OOM, "tr_create: host allocation failed");
    c->device = config->device;
    c->width = config->width;
    c->height = config->height;
    c->band_y0 = config->band_y1 ? config->band_y0 : 0;
    c->band_y1 = config->band_y1 ? config->band_y1 : config->height;
    c->flags = config->flags;
    if (c->band_y0 >= c->band_y1 || c->band_y1 > c->height) {
        delete c;
        return fail(TR_ERR_INVALID_ARG, "tr_create: band [%u,%u) outside the frame", config->band_y0, config->band_y1);
    }
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, c->device) == cudaSuccess) c->sm_count = prop.multiProcessorCount;
    e = cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) {
        delete c;
        return fail(TR_ERR_CUDA, "cudaStreamCreate: %s", cudaGetErrorString(e));
    }
    c->stream = c->own_stream;
    int32_t s = alloc_frame(c);
    if (s != TR_OK) {
        tr_destroy(c);
        return s;
    }
    *out_ctx = c;
    return TR_OK;
}

int32_t tr_destroy(tr_ctx* c) {
    if (!c) return TR_OK;
    TR_NOT_GROUPED(c, "tr_destroy", "tr_group_destroy first");
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    comm_release(c);
    DevBuf* bufs[] = {&c->instances, &c->instances_alt, &c->lights_alt, &c->primitives, &c->materials, &c->lights, &c->lut, &c->mesh_pos, &c->mesh_nrm,
                      &c->mesh_uv, &c->mesh_idx, &c->visible_ids, &c->cull_scalars, &c->draws[0], &c->draws[1],
                      &c->draws[2], &c->draws[3], &c->work_prefix, &c->slot_z, &c->slot_first, &c->block_entry, &c->chunk_spheres, &c->prim_chunk_base, &c->cluster_aabbs, &c->cluster_counts,
                      &c->cluster_indices, &c->vis[0], &c->vis[1], &c->bin_entries, &c->bin_state, &c->tri_records, &c->dev_status, &c->band_list, &c->hdr, &c->hdr_f32, &c->pyramid,
                      &c->srgb8, &c->mip_counter, &c->shade_counter, &c->accel_tlas, &c->accel_blas, &c->accel_inst, &c->accel_tris,
                      &c->accel_prim_table, &c->accel_scratch, &c->accel_build_scratch, &c->accel_refit, &c->shadow_mask[0], &c->shadow_mask[1], &c->transform_staging};
    for (DevBuf* b : bufs) b->release();
    for (DevBuf& b : c->tex_data) b.release();
    c->tex_table.release();
    c->tex_tables.release();
    for (int l = 0; l < 2; l++) {
        GLayer& g = c->layer[l];
        g.depth.release(); g.normal.release(); g.uv.release(); g.material_id.release(); g.scale.release(); g.position.release();
        g.duv.release(); g.ddepth.release();
    }
    if (c->ev_begin) {
        for (int f = 0; f < kTimingRing; f++)
            for (int i = 0; i < P_COUNT; i++) {
                cudaEventDestroy(c->ev_begin[f][i]);
                cudaEventDestroy(c->ev_end[f][i]);
            }
        delete[] c->ev_begin;
        delete[] c->ev_end;
        delete[] c->ev_used;
    }
    if (c->upload_stream) {
        cudaStreamSynchronize(c->upload_stream);
        cudaStreamDestroy(c->upload_stream);
    }
    if (c->side_stream) {
        cudaStreamSynchronize(c->side_stream);
        cudaStreamDestroy(c->side_stream);
        cudaEventDestroy(c->ev_fork);
        cudaEventDestroy(c->ev_join);
    }
    for (cudaEvent_t e : {c->ev_frame_begin, c->ev_inst_ready, c->ev_lights_ready})
        if (e) cudaEventDestroy(e);
    if (c->copy_stream) {
        cudaStreamSynchronize(c->copy_stream);
        cudaStreamDestroy(c->copy_stream);
        cudaEventDestroy(c->ev_frame_done);
        cudaEventDestroy(c->ev_copy_done);
    }
    if (c->own_stream) cudaStreamDestroy(c->own_stream);
    delete c;
    return TR_OK;
}

int32_t tr_resize(tr_ctx* c, uint32_t width, uint32_t height) {
    TR_CHECK_CTX(c);
    TR_NOT_GROUPED(c, "tr_resize", "tr_group_resize");
    if (width == 0 || height == 0) return fail(TR_ERR_INVALID_ARG, "tr_resize: empty framebuffer");
    TR_CUDA(cudaStreamSynchronize(c->stream));
    if (c->peers_attached) return fail(TR_ERR_STATE, "tr_resize: detach the peer mappings first (tr_comm_destroy); they name the old frame buffers");
    return resize_frame(c, width, height);
}

int32_t tr_set_band(tr_ctx* c, uint32_t y0, uint32_t y1) {
    TR_CHECK_CTX(c);
    TR_NOT_GROUPED(c, "tr_set_band", "tr_group_set_bands");
    if (y0 >= y1 || y1 > c->height) return fail(TR_ERR_INVALID_ARG, "tr_set_band: [%u,%u) outside the frame", y0, y1);
    c->band_y0 = y0;
    c->band_y1 = y1;
    return TR_OK;
}

int32_t tr_set_stream(tr_ctx* c, void* cuda_stream) {
    TR_CHECK_CTX(c);
    c->stream = cuda_stream ? reinterpret_cast<cudaStream_t>(cuda_stream) : c->own_stream;
    return TR_OK;
}

int32_t tr_sync(tr_ctx* c) {
    TR_CHECK_CTX(c);
    TR_CUDA(cudaStreamSynchronize(c->stream));
    if (c->copy_stream) TR_CUDA(cudaStreamSynchronize(c->copy_stream));
    return check_device_status(c, "tr_sync");
}

// ------------------------------------------------------------------ uploads
// Where a source of tr_update_mesh_vertices / tr_set_lights / tr_update_instance_transforms lives.  kLocal: memory a
// kernel on the context's device may read in place (its own device memory, managed memory); kPeer: another device's memory,
// which only a copy reads (peer access may be off).  Both device kinds are read on the context stream, in stream order.
enum SourceKind { kHost, kLocal, kPeer };
static SourceKind source_kind(const tr_ctx* c, const void* p) {
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, p) != cudaSuccess) {
        cudaGetLastError();
        return kHost;
    }
    if (attr.type == cudaMemoryTypeManaged) return kLocal;
    if (attr.type == cudaMemoryTypeDevice) return attr.device == c->device ? kLocal : kPeer;
    return kHost;
}

static int32_t upload(tr_ctx* c, DevBuf& b, const void* src, size_t bytes, cudaMemcpyKind kind = cudaMemcpyHostToDevice) {
    TR_TRY(b.ensure(bytes));
    if (bytes) TR_CUDA(cudaMemcpyAsync(b.p, src, bytes, kind, c->stream));
    return TR_OK;
}

// An upload that may run ahead (see tr_internal.h).  Taken when the source is page-locked, a frame has been enqueued, and this
// buffer has not been uploaded since: `alt` was read last by the frame before the enqueued one, so it is free once the
// enqueued frame has BEGUN (ev_frame_begin, recorded at the top of tr_frame).  Otherwise the copy goes into the compute stream.
static int32_t upload_ahead(tr_ctx* c, DevBuf& cur, DevBuf& alt, bool& uploaded, cudaEvent_t& ev_ready, const void* src, size_t bytes) {
    cudaPointerAttributes attr;
    const bool pinned = bytes && cudaPointerGetAttributes(&attr, src) == cudaSuccess && attr.type == cudaMemoryTypeHost;
    if (!pinned) cudaGetLastError();
    if (!pinned || !c->frame_begin_valid || uploaded) return upload(c, cur, src, bytes);
    if (!c->upload_stream) TR_CUDA(cudaStreamCreateWithFlags(&c->upload_stream, cudaStreamNonBlocking));
    if (!ev_ready) TR_CUDA(cudaEventCreateWithFlags(&ev_ready, cudaEventDisableTiming));
    TR_TRY(alt.ensure(bytes));
    TR_CUDA(cudaStreamWaitEvent(c->upload_stream, c->ev_frame_begin, 0));
    TR_CUDA(cudaMemcpyAsync(alt.p, src, bytes, cudaMemcpyHostToDevice, c->upload_stream));
    TR_CUDA(cudaEventRecord(ev_ready, c->upload_stream));
    TR_CUDA(cudaStreamWaitEvent(c->stream, ev_ready, 0));   // everything enqueued from here on sees the new contents
    std::swap(cur, alt);
    uploaded = true;
    return TR_OK;
}

int32_t tr_set_instances(tr_ctx* c, const tr_instance* instances, uint32_t n) {
    TR_CHECK_CTX(c);
    if (n && !instances) return fail(TR_ERR_INVALID_ARG, "tr_set_instances: null");
    if (n >= (1u << 24)) return fail(TR_ERR_UNSUPPORTED, "tr_set_instances: at most 2^24-1 instances");
    TR_TRY(upload_ahead(c, c->instances, c->instances_alt, c->inst_uploaded, c->ev_inst_ready, instances, (size_t)n * sizeof(tr_instance)));
    c->n_instances = n;
    c->h_inst_prim.resize(n);
    c->h_inst_mat.resize(n);
    for (uint32_t i = 0; i < n; i++) {
        c->h_inst_prim[i] = instances[i].primitive_id;
        c->h_inst_mat[i] = instances[i].material_id;
    }
    c->scene_checked = false;
    c->tri_bound_valid = false;
    c->cull_valid = false;
    c->accel_tlas_valid = false;  // src/main.rs:1263-1345: an instance write is followed by a top-level update
    return TR_OK;
}

// Only the transforms move, so nothing the host holds about the instances changes (ids, the triangle bound, the top-level
// count, validate_scene).  A source the kernel may read in place (device memory of this device, 16-byte aligned) is
// scattered straight into the instance buffer; any other one is first copied contiguously into the staging buffer, on the
// same stream: one copy of n * 32 bytes, where a 2D copy of 32-byte rows straight into the records would crawl over PCIe.
int32_t tr_update_instance_transforms(tr_ctx* c, uint32_t first, uint32_t n, const tr_packed_similarity* transforms) {
    TR_CHECK_CTX(c);
    if ((uint64_t)first + n > c->n_instances)
        return fail(TR_ERR_INVALID_ARG, "tr_update_instance_transforms: instances [%u, %u + %u) of %u", first, first, n, c->n_instances);
    if (n == 0) return TR_OK;
    if (!transforms) return fail(TR_ERR_INVALID_ARG, "tr_update_instance_transforms: null");
    const SourceKind kind = source_kind(c, transforms);
    const tr_packed_similarity* src = transforms;
    if (kind != kLocal || ((uintptr_t)transforms & 15u)) {
        const size_t bytes = (size_t)n * sizeof(tr_packed_similarity);
        TR_TRY(upload(c, c->transform_staging, transforms, bytes, kind == kHost ? cudaMemcpyHostToDevice : cudaMemcpyDefault));
        src = c->transform_staging.as<tr_packed_similarity>();
    }
    TR_TRY(launch_instance_transforms(c, first, n, src));
    c->cull_valid = false;
    c->accel_tlas_valid = false;   // as after tr_set_instances: the top level needs an update before the next traced frame
    return TR_OK;
}

int32_t tr_set_primitives(tr_ctx* c, const tr_primitive_info* prims, uint32_t n) {
    TR_CHECK_CTX(c);
    if (n && !prims) return fail(TR_ERR_INVALID_ARG, "tr_set_primitives: null");
    bool clip = false;
    for (uint32_t i = 0; i < n; i++) {
        if (prims[i].draw_buffer_index > 3)
            return fail(TR_ERR_INVALID_ARG, "tr_set_primitives: primitive %u names draw buffer %u (0..3)", i, prims[i].draw_buffer_index);
        clip = clip || (prims[i].draw_buffer_index & 1u);
    }
    c->prims_alpha_clip = clip;
    c->chunks_valid = false;
    TR_TRY(upload(c, c->primitives, prims, (size_t)n * sizeof(tr_primitive_info)));
    c->n_primitives = n;
    c->h_prim_tris.resize(n);
    c->h_prim_first.resize(n);
    c->h_prim_count.resize(n);
    c->h_prim_bucket.resize(n);
    for (uint32_t i = 0; i < n; i++) {
        c->h_prim_tris[i] = prims[i].index_count / 3u;
        c->h_prim_first[i] = prims[i].first_index;
        c->h_prim_count[i] = prims[i].index_count;
        c->h_prim_bucket[i] = prims[i].draw_buffer_index;
    }
    c->scene_checked = false;
    c->tri_bound_valid = false;
    c->cull_valid = false;
    c->accel_blas_valid = c->accel_tlas_valid = false;
    return TR_OK;
}

int32_t tr_set_materials(tr_ctx* c, const tr_material_info* materials, uint32_t n) {
    TR_CHECK_CTX(c);
    if (n && !materials) return fail(TR_ERR_INVALID_ARG, "tr_set_materials: null");
    bool textured = false;
    for (uint32_t i = 0; i < n; i++) {
        const int32_t* t = &materials[i].textures.diffuse;
        for (int k = 0; k < 9; k++) {
            if (t[k] < -1 || t[k] >= (int32_t)TR_MAX_IMAGES)
                return fail(TR_ERR_INVALID_ARG, "tr_set_materials: material %u texture slot %d names image %d (0..%u or -1)", i, k, t[k], TR_MAX_IMAGES - 1);
            if (k != 4 && t[k] != -1) textured = true;  // slot 4 (occlusion) is never sampled by the shaders
        }
    }
    c->materials_textured = textured;
    TR_TRY(upload(c, c->materials, materials, (size_t)n * sizeof(tr_material_info)));
    c->n_materials = n;
    c->scene_checked = false;
    return TR_OK;
}

int32_t tr_set_lights(tr_ctx* c, const tr_light* lights, uint32_t n) {
    TR_CHECK_CTX(c);
    if (n && !lights) return fail(TR_ERR_INVALID_ARG, "tr_set_lights: null");
    // A device source is copied on the context stream, after whatever produced it there, into the buffer the next frame
    // reads: behind a run-ahead upload of this frame too, since the context stream already waits for that copy.
    if (n && source_kind(c, lights) != kHost)
        TR_TRY(upload(c, c->lights, lights, (size_t)n * sizeof(tr_light), cudaMemcpyDefault));
    else
        TR_TRY(upload_ahead(c, c->lights, c->lights_alt, c->lights_uploaded, c->ev_lights_ready, lights, (size_t)n * sizeof(tr_light)));
    c->n_lights = n;
    c->cluster_lights_valid = false;
    return TR_OK;
}

int32_t tr_set_uniforms(tr_ctx* c, const tr_uniforms* u) {
    TR_CHECK_CTX(c);
    if (!u) return fail(TR_ERR_INVALID_ARG, "tr_set_uniforms: null");
    if (u->debug_clusters != 0) return fail(TR_ERR_UNSUPPORTED, "tr_set_uniforms: debug_clusters must be 0");
    const uint64_t n = (uint64_t)u->num_clusters.x * u->num_clusters.y * u->light_clustering_coefficients.num_depth_slices;
    if (n == 0 || n > (1u << 24)) return fail(TR_ERR_INVALID_ARG, "tr_set_uniforms: bad cluster grid");
    if ((uint32_t)n != c->n_clusters) c->clusters_valid = c->cluster_lights_valid = false;
    c->uniforms = *u;
    c->n_clusters = (uint32_t)n;
    c->have_uniforms = true;
    return TR_OK;
}

int32_t tr_set_ggx_lut(tr_ctx* c, const uint8_t* rgba8, uint32_t width, uint32_t height) {
    TR_CHECK_CTX(c);
    if (!rgba8 || !width || !height) return fail(TR_ERR_INVALID_ARG, "tr_set_ggx_lut: null/empty");
    std::vector<uint8_t> rg((size_t)width * height * 2);  // only .xy is ever sampled (shader lib.rs:126-133)
    for (size_t i = 0; i < (size_t)width * height; i++) {
        rg[i * 2] = rgba8[i * 4];
        rg[i * 2 + 1] = rgba8[i * 4 + 1];
    }
    TR_CUDA(cudaStreamSynchronize(c->stream));  // a frame in flight may still sample the old table (as tr_set_texture does)
    TR_TRY(c->lut.ensure(rg.size()));
    TR_CUDA(cudaMemcpyAsync(c->lut.p, rg.data(), rg.size(), cudaMemcpyHostToDevice, c->stream));
    TR_CUDA(cudaStreamSynchronize(c->stream));  // `rg` is a local
    c->lut_w = width;
    c->lut_h = height;
    return TR_OK;
}

// Level texel offsets of an image (TexDesc.off) and its texel count over those levels.
static size_t texture_layout(trd::TexDesc* d, uint32_t width, uint32_t height, uint32_t n_levels, int32_t srgb) {
    d->w = width;
    d->h = height;
    d->levels = n_levels;
    d->srgb = srgb ? 1u : 0u;
    size_t total = 0;
    for (uint32_t l = 0; l < n_levels; l++) {
        d->off[l] = (uint32_t)total;
        const uint32_t w = width >> l ? width >> l : 1u, h = height >> l ? height >> l : 1u;
        total += (size_t)w * h;
    }
    return total;
}

static size_t texture_texels(const trd::TexDesc& d) {
    const uint32_t l = d.levels - 1, w = d.w >> l ? d.w >> l : 1u, h = d.h >> l ? d.h >> l : 1u;
    return (size_t)d.off[l] + (size_t)w * h;
}

static void bind_texture(tr_ctx* c, uint32_t index, trd::TexDesc d, bool chain) {
    d.base = c->tex_data[index].as<float4>();
    c->h_tex[index] = d;
    c->tex_chain[index] = chain;
    if (index + 1 > c->n_textures) c->n_textures = index + 1;
    c->tex_table_dirty = true;
}

// At least `need` bytes for image `index`, in stream order where it can be: a first bind allocates on the context stream
// (unlike cudaMalloc, a stream-ordered allocation never waits for the device to reclaim freed memory); an allocation that
// must grow waits for the frame in flight, which may still sample the old image.  The first bind takes the device's default
// pool by name, whatever pool the host made current: that is the pool tr_group_create opens to the other members' devices
// (peer access to pool memory follows cudaMemPoolSetAccess, not cudaDeviceEnablePeerAccess).
static int32_t ensure_texture(tr_ctx* c, uint32_t index, size_t need) {
    DevBuf& buf = c->tex_data[index];
    if (buf.p && buf.bytes < need) TR_CUDA(cudaStreamSynchronize(c->stream));
    if (!buf.p) {
        cudaMemPool_t pool;
        TR_CUDA(cudaDeviceGetDefaultMemPool(&pool, c->device));
        TR_CUDA(cudaMallocFromPoolAsync(&buf.p, need, pool, c->stream));
        buf.bytes = need;
    }
    return buf.ensure(need);
}

int32_t tr_set_texture(tr_ctx* c, uint32_t index, const uint8_t* const* levels, uint32_t n_levels, uint32_t width, uint32_t height,
                       int32_t srgb) {
    TR_CHECK_CTX(c);
    if (index >= TR_MAX_IMAGES) return fail(TR_ERR_INVALID_ARG, "tr_set_texture: image %u of at most %u", index, TR_MAX_IMAGES);
    if (!levels || n_levels == 0 || n_levels > 16 || !width || !height) return fail(TR_ERR_INVALID_ARG, "tr_set_texture: bad arguments");
    const TexTables& tab = texture_tables();
    const float* table = tab.dec32[srgb ? 0 : 1];   // sRGB8 -> linear, evaluated in double and rounded once
    const float* unorm = tab.dec32[1];              // alpha stays linear in the sRGB formats
    trd::TexDesc d{};
    for (uint32_t l = 0; l < n_levels; l++)
        if (!levels[l]) return fail(TR_ERR_INVALID_ARG, "tr_set_texture: level %u is null", l);
    const size_t total = texture_layout(&d, width, height, n_levels, srgb);
    std::vector<float> texels(total * 4);
    for (uint32_t l = 0; l < n_levels; l++) {
        const uint32_t w = width >> l ? width >> l : 1u, h = height >> l ? height >> l : 1u;
        const uint8_t* src = levels[l];
        float* dst = texels.data() + (size_t)d.off[l] * 4;
        for (size_t i = 0; i < (size_t)w * h; i++) {
            dst[i * 4 + 0] = table[src[i * 4 + 0]];
            dst[i * 4 + 1] = table[src[i * 4 + 1]];
            dst[i * 4 + 2] = table[src[i * 4 + 2]];
            dst[i * 4 + 3] = unorm[src[i * 4 + 3]];
        }
    }
    TR_CUDA(cudaStreamSynchronize(c->stream));  // a frame in flight may still sample the old image
    TR_TRY(c->tex_data[index].ensure(total * 16));
    TR_CUDA(cudaMemcpy(c->tex_data[index].p, texels.data(), total * 16, cudaMemcpyHostToDevice));
    bind_texture(c, index, d, false);
    return TR_OK;
}

// Level 0 as RGBA8 into the byte chain behind the image's texels, then the device builds the store and the rest of the chain
// (k_textures.cu), all in stream order.  The allocation is the image's own: a rebind that fits it reuses it without a wait,
// since every frame that may still read the old texels was enqueued before the kernels that overwrite them.
int32_t tr_set_texture_async(tr_ctx* c, uint32_t index, const uint8_t* rgba8, uint32_t width, uint32_t height, int32_t srgb,
                             uint32_t n_levels) {
    TR_CHECK_CTX(c);
    if (index >= TR_MAX_IMAGES) return fail(TR_ERR_INVALID_ARG, "tr_set_texture_async: image %u of at most %u", index, TR_MAX_IMAGES);
    if (!rgba8 || !width || !height || n_levels > 16) return fail(TR_ERR_INVALID_ARG, "tr_set_texture_async: bad arguments");
    const uint32_t full = mip_levels_for_size(width, height);
    if (n_levels > full || (n_levels == 0 && full > 16))
        return fail(TR_ERR_INVALID_ARG, "tr_set_texture_async: %u levels for a %ux%u image (full chain %u, at most 16)",
                    n_levels ? n_levels : full, width, height, full);
    trd::TexDesc d{};
    const size_t total = texture_layout(&d, width, height, n_levels ? n_levels : full, srgb);
    if (total > 0xffffffffull) return fail(TR_ERR_UNSUPPORTED, "tr_set_texture_async: more than 2^32 texels");
    const size_t need = total * 20;   // RGBA32F texels, then the RGBA8 bytes of every level
    if (!c->tex_tables.p) {
        TR_TRY(c->tex_tables.ensure(sizeof(TexTables)));
        TR_CUDA(cudaMemcpyAsync(c->tex_tables.p, &texture_tables(), sizeof(TexTables), cudaMemcpyHostToDevice, c->stream));
    }
    TR_TRY(ensure_texture(c, index, need));
    DevBuf& buf = c->tex_data[index];
    uint8_t* chain = buf.as<uint8_t>() + total * 16;
    TR_CUDA(cudaMemcpyAsync(chain, rgba8, (size_t)width * height * 4, cudaMemcpyHostToDevice, c->stream));
    d.base = buf.as<float4>();
    TR_TRY(launch_texture_chain(c->tex_tables.as<TexTables>(), d, chain, c->sm_count, c->stream));
    bind_texture(c, index, d, true);
    return TR_OK;
}

int32_t tr_set_mesh(tr_ctx* c, const float* positions, const float* normals, const float* uvs, uint32_t n_vertices,
                    const uint32_t* indices, uint32_t n_indices) {
    TR_CHECK_CTX(c);
    if (!positions || !normals || !uvs || !indices) return fail(TR_ERR_INVALID_ARG, "tr_set_mesh: null");
    for (uint32_t i = 0; i < n_indices; i++)
        if (indices[i] >= n_vertices) return fail(TR_ERR_INVALID_ARG, "tr_set_mesh: index %u out of range", i);
    TR_TRY(upload(c, c->mesh_pos, positions, (size_t)n_vertices * 12));
    TR_TRY(upload(c, c->mesh_nrm, normals, (size_t)n_vertices * 12));
    TR_TRY(upload(c, c->mesh_uv, uvs, (size_t)n_vertices * 8));
    TR_TRY(upload(c, c->mesh_idx, indices, (size_t)n_indices * 4));
    c->n_vertices = n_vertices;
    c->n_indices = n_indices;
    c->chunks_valid = false;
    c->scene_checked = false;
    c->accel_blas_valid = c->accel_tlas_valid = false;
    return TR_OK;
}

// Vertex animation: the positions and normals of [first_vertex, first_vertex + n) in stream order on the context stream (not
// the run-ahead upload stream: the frame in flight reads these buffers), then everything that depends on the positions, on
// the device: the chunk spheres and, once built, the bottom-level trees (refit; the top level needs an update after it).
int32_t tr_update_mesh_vertices(tr_ctx* c, uint32_t first_vertex, uint32_t n, const float* positions, const float* normals) {
    TR_CHECK_CTX(c);
    if (!c->mesh_pos.p) return fail(TR_ERR_STATE, "tr_update_mesh_vertices: no mesh (tr_set_mesh)");
    if ((uint64_t)first_vertex + n > c->n_vertices)
        return fail(TR_ERR_INVALID_ARG, "tr_update_mesh_vertices: vertices [%u, %u + %u) of %u", first_vertex, first_vertex, n, c->n_vertices);
    if (n == 0) return TR_OK;
    if (!positions || !normals) return fail(TR_ERR_INVALID_ARG, "tr_update_mesh_vertices: null");
    const cudaMemcpyKind pk = source_kind(c, positions) == kHost ? cudaMemcpyHostToDevice : cudaMemcpyDefault;
    const cudaMemcpyKind nk = source_kind(c, normals) == kHost ? cudaMemcpyHostToDevice : cudaMemcpyDefault;
    TR_CUDA(cudaMemcpyAsync(c->mesh_pos.as<float>() + (size_t)first_vertex * 3, positions, (size_t)n * 12, pk, c->stream));
    TR_CUDA(cudaMemcpyAsync(c->mesh_nrm.as<float>() + (size_t)first_vertex * 3, normals, (size_t)n * 12, nk, c->stream));
    if (c->chunks_valid) TR_TRY(launch_chunk_spheres(c));
    else TR_TRY(ensure_chunks(c));
    if (c->accel_blas_valid) {
        TR_TRY(accel_refit_blas(c));
        c->accel_tlas_valid = false;   // the top level holds the old primitive boxes: it needs an update, as after tr_set_instances
    }
    return TR_OK;
}

int32_t tr_read_chunk_spheres(tr_ctx* c, float* spheres, uint32_t capacity, uint32_t* n_spheres) {
    TR_CHECK_CTX(c);
    TR_TRY(ensure_chunks(c));
    const uint32_t n = c->n_chunks;
    if (n_spheres) *n_spheres = n;
    if (spheres && capacity < n) return fail(TR_ERR_INVALID_ARG, "tr_read_chunk_spheres: capacity %u < %u", capacity, n);
    if (spheres && n) TR_CUDA(cudaMemcpyAsync(spheres, c->chunk_spheres.p, (size_t)n * 16, cudaMemcpyDeviceToHost, c->stream));
    TR_CUDA(cudaStreamSynchronize(c->stream));
    return TR_OK;
}

}  // extern "C"

// ------------------------------------------------------------------ scene replication (tr_group_replicate_scene)
// The host state of an empty scene: no counts, no bound image, nothing valid that a frame or a build would read.  The
// device buffers stay allocated (grow-only).
static void clear_scene(tr_ctx* c) {
    c->n_vertices = c->n_indices = c->n_primitives = c->n_materials = c->n_instances = c->n_lights = 0;
    c->have_uniforms = c->clusters_valid = c->cluster_lights_valid = false;
    c->lut_w = c->lut_h = 0;
    c->prims_alpha_clip = c->materials_textured = false;
    for (uint32_t i = 0; i < TR_MAX_IMAGES; i++) {
        c->h_tex[i] = trd::TexDesc{};
        c->tex_chain[i] = false;
    }
    c->n_textures = 0;
    c->tex_table_dirty = true;
    for (std::vector<uint32_t>* v : {&c->h_prim_tris, &c->h_inst_prim, &c->h_inst_mat, &c->h_prim_first, &c->h_prim_count,
                                     &c->h_chunk_base, &c->h_prim_root, &c->h_prim_tri_base, &c->h_prim_bucket})
        v->clear();
    c->n_chunks = 0;
    c->chunks_valid = c->chunk_cull = false;
    c->scene_checked = c->tri_bound_valid = c->cull_valid = false;
    c->max_triangles = 0;
    c->accel_blas_nodes = c->accel_n_tris = c->accel_n_instances = 0;
    c->accel_blas_valid = c->accel_tlas_valid = false;
}

// One destination: every device buffer a frame reads is copied byte for byte on dst's stream (cudaMemcpyDefault: a peer
// device or the same one), and the host state that describes those buffers is copied on the host, so dst ends as a context
// that received the same uploads and builds.  The trees hold node and triangle indices, never pointers, so they are valid
// at dst's addresses as they are; the texture descriptors hold absolute bases, so dst's table is rebuilt.  What is dst's
// own stays: frame targets, G-buffers, shadow masks, light lists, cull outputs, timers, streams, scratch and the run-ahead
// bookkeeping.  dst's host state is first set to an empty scene: a buffer that grows is freed before it is reallocated, so
// a failure part-way (an allocation) leaves dst empty, to be loaded again, and never describing memory it no longer owns.
int32_t tr::replicate_scene(tr_ctx* dst, const tr_ctx* src) {
    const cudaMemcpyKind k = cudaMemcpyDefault;
    clear_scene(dst);
    TR_TRY(upload(dst, dst->mesh_pos, src->mesh_pos.p, (size_t)src->n_vertices * 12, k));
    TR_TRY(upload(dst, dst->mesh_nrm, src->mesh_nrm.p, (size_t)src->n_vertices * 12, k));
    TR_TRY(upload(dst, dst->mesh_uv, src->mesh_uv.p, (size_t)src->n_vertices * 8, k));
    TR_TRY(upload(dst, dst->mesh_idx, src->mesh_idx.p, (size_t)src->n_indices * 4, k));
    TR_TRY(upload(dst, dst->primitives, src->primitives.p, (size_t)src->n_primitives * sizeof(tr_primitive_info), k));
    TR_TRY(upload(dst, dst->materials, src->materials.p, (size_t)src->n_materials * sizeof(tr_material_info), k));
    TR_TRY(upload(dst, dst->instances, src->instances.p, (size_t)src->n_instances * sizeof(tr_instance), k));
    TR_TRY(upload(dst, dst->lights, src->lights.p, (size_t)src->n_lights * sizeof(tr_light), k));
    if (src->lut_w) TR_TRY(upload(dst, dst->lut, src->lut.p, (size_t)src->lut_w * src->lut_h * 2, k));
    if (src->clusters_valid)
        TR_TRY(upload(dst, dst->cluster_aabbs, src->cluster_aabbs.p, (size_t)src->n_clusters * sizeof(tr_cluster_aabb), k));
    if (src->chunks_valid) {
        TR_TRY(upload(dst, dst->prim_chunk_base, src->prim_chunk_base.p, src->h_chunk_base.size() * 4, k));
        TR_TRY(upload(dst, dst->chunk_spheres, src->chunk_spheres.p, (size_t)src->n_chunks * 16, k));
    }
    if (src->accel_blas_valid) {
        const size_t nn = src->accel_blas_nodes, nt = src->accel_n_tris;
        TR_TRY(upload(dst, dst->accel_blas, src->accel_blas.p, nn * sizeof(trd::AccelNode), k));
        TR_TRY(upload(dst, dst->accel_tris, src->accel_tris.p, nt * 3 * sizeof(float4), k));
        TR_TRY(upload(dst, dst->accel_prim_table, src->accel_prim_table.p, (size_t)src->n_primitives * sizeof(trd::TlasPrim), k));
        TR_TRY(upload(dst, dst->accel_refit, src->accel_refit.p, (nn * 2 + nt) * 4, k));   // parents, arrivals, triangle sources
        if (src->accel_tlas_valid) {
            const size_t m = src->accel_n_instances;
            TR_TRY(upload(dst, dst->accel_tlas, src->accel_tlas.p, (m >= 2 ? m - 1 : 1) * sizeof(trd::AccelNode), k));
            TR_TRY(upload(dst, dst->accel_inst, src->accel_inst.p, m * sizeof(trd::AccelInstance), k));
        }
    }
    for (uint32_t i = 0; i < src->n_textures; i++) {   // an image unbound on the source stays unbound here (clear_scene)
        const trd::TexDesc& d = src->h_tex[i];
        if (!d.base) continue;
        const size_t bytes = texture_texels(d) * (src->tex_chain[i] ? 20 : 16);
        TR_TRY(ensure_texture(dst, i, bytes));
        TR_CUDA(cudaMemcpyAsync(dst->tex_data[i].p, src->tex_data[i].p, bytes, k, dst->stream));
        bind_texture(dst, i, d, src->tex_chain[i]);
    }
    dst->n_textures = src->n_textures;
    dst->tex_table_dirty = true;

    dst->n_vertices = src->n_vertices;
    dst->n_indices = src->n_indices;
    dst->n_primitives = src->n_primitives;
    dst->n_materials = src->n_materials;
    dst->n_instances = src->n_instances;
    dst->n_lights = src->n_lights;
    dst->uniforms = src->uniforms;
    dst->have_uniforms = src->have_uniforms;
    dst->n_clusters = src->n_clusters;
    dst->clusters_valid = src->clusters_valid;
    dst->cluster_lights_valid = false;   // as after tr_set_lights: the next frame assigns the new lights
    dst->lut_w = src->lut_w;
    dst->lut_h = src->lut_h;
    dst->prims_alpha_clip = src->prims_alpha_clip;
    dst->materials_textured = src->materials_textured;
    dst->h_prim_tris = src->h_prim_tris;
    dst->h_inst_prim = src->h_inst_prim;
    dst->h_inst_mat = src->h_inst_mat;
    dst->h_prim_first = src->h_prim_first;
    dst->h_prim_count = src->h_prim_count;
    dst->h_chunk_base = src->h_chunk_base;
    dst->n_chunks = src->n_chunks;
    dst->chunks_valid = src->chunks_valid;
    dst->chunk_cull = src->chunk_cull;
    dst->scene_checked = src->scene_checked;
    dst->max_triangles = src->max_triangles;
    dst->tri_bound_valid = src->tri_bound_valid;
    dst->cull_valid = false;
    dst->h_prim_root = src->h_prim_root;
    dst->h_prim_tri_base = src->h_prim_tri_base;
    dst->h_prim_bucket = src->h_prim_bucket;
    dst->accel_blas_nodes = src->accel_blas_nodes;
    dst->accel_n_tris = src->accel_n_tris;
    dst->accel_n_instances = src->accel_n_instances;
    dst->accel_blas_valid = src->accel_blas_valid;
    dst->accel_tlas_valid = src->accel_blas_valid && src->accel_tlas_valid;
    return TR_OK;
}

extern "C" {

// ------------------------------------------------------------------ ray-queried shadows
int32_t tr_build_acceleration_structures(tr_ctx* c, uint64_t* address) {
    TR_CHECK_CTX(c);
    if (!address) return fail(TR_ERR_INVALID_ARG, "tr_build_acceleration_structures: null");
    *address = 0;
    TR_TRY(accel_build(c));
    *address = (uint64_t)(uintptr_t)c->accel_tlas.p;
    return TR_OK;
}

int32_t tr_build_acceleration_structures_async(tr_ctx* c, uint64_t* address) {
    TR_CHECK_CTX(c);
    if (!address) return fail(TR_ERR_INVALID_ARG, "tr_build_acceleration_structures_async: null");
    *address = 0;
    TR_TRY(accel_build_async(c));
    *address = (uint64_t)(uintptr_t)c->accel_tlas.p;
    return TR_OK;
}

int32_t tr_update_top_level_acceleration_structure(tr_ctx* c, uint64_t* address) {
    TR_CHECK_CTX(c);
    TR_TRY(accel_build_tlas(c));
    if (address) *address = (uint64_t)(uintptr_t)c->accel_tlas.p;
    return TR_OK;
}

int32_t tr_update_top_level_acceleration_structure_async(tr_ctx* c, uint64_t* address) {
    TR_CHECK_CTX(c);
    TR_TRY(accel_build_tlas_async(c));
    if (address) *address = (uint64_t)(uintptr_t)c->accel_tlas.p;
    return TR_OK;
}

int32_t tr_read_top_level_acceleration_structure(tr_ctx* c, void* nodes, uint32_t node_capacity, uint32_t* n_nodes, void* instances,
                                                 uint32_t instance_capacity, uint32_t* n_instances) {
    TR_CHECK_CTX(c);
    if (!c->accel_blas_valid || !c->accel_tlas_valid)
        return fail(TR_ERR_STATE, "tr_read_top_level_acceleration_structure: acceleration structures not built");
    const uint32_t m = c->accel_n_instances, nn = m >= 2 ? m - 1 : 1;   // a binary tree over m leaves, or the one root
    if (n_nodes) *n_nodes = nn;
    if (n_instances) *n_instances = m;
    if ((nodes && node_capacity < nn) || (instances && instance_capacity < m))
        return fail(TR_ERR_INVALID_ARG, "tr_read_top_level_acceleration_structure: capacity %u nodes / %u instances < %u / %u",
                    node_capacity, instance_capacity, nn, m);
    if (nodes) TR_CUDA(cudaMemcpyAsync(nodes, c->accel_tlas.p, (size_t)nn * sizeof(trd::AccelNode), cudaMemcpyDeviceToHost, c->stream));
    if (instances && m)
        TR_CUDA(cudaMemcpyAsync(instances, c->accel_inst.p, (size_t)m * sizeof(trd::AccelInstance), cudaMemcpyDeviceToHost, c->stream));
    TR_CUDA(cudaStreamSynchronize(c->stream));
    return TR_OK;
}

int32_t tr_read_bottom_level_acceleration_structures(tr_ctx* c, void* nodes, uint32_t node_capacity, uint32_t* n_nodes, void* tris,
                                                     uint32_t tri_capacity, uint32_t* n_tris) {
    TR_CHECK_CTX(c);
    if (!c->accel_blas_valid)
        return fail(TR_ERR_STATE, "tr_read_bottom_level_acceleration_structures: acceleration structures not built");
    const uint32_t nn = c->accel_blas_nodes, nt = c->accel_n_tris;
    if (n_nodes) *n_nodes = nn;
    if (n_tris) *n_tris = nt;
    if ((nodes && node_capacity < nn) || (tris && tri_capacity < nt))
        return fail(TR_ERR_INVALID_ARG, "tr_read_bottom_level_acceleration_structures: capacity %u nodes / %u triangles < %u / %u",
                    node_capacity, tri_capacity, nn, nt);
    if (nodes && nn) TR_CUDA(cudaMemcpyAsync(nodes, c->accel_blas.p, (size_t)nn * sizeof(trd::AccelNode), cudaMemcpyDeviceToHost, c->stream));
    if (tris && nt) TR_CUDA(cudaMemcpyAsync(tris, c->accel_tris.p, (size_t)nt * 3 * sizeof(float4), cudaMemcpyDeviceToHost, c->stream));
    TR_CUDA(cudaStreamSynchronize(c->stream));
    return TR_OK;
}

int32_t tr_trace_shadow_rays(tr_ctx* c, uint32_t n, const float* origins, const float* directions, const float* t_max, uint8_t* lit) {
    TR_CHECK_CTX(c);
    if (!c->accel_blas_valid || !c->accel_tlas_valid) return fail(TR_ERR_STATE, "tr_trace_shadow_rays: acceleration structures not built");
    if (n && (!origins || !directions || !t_max || !lit)) return fail(TR_ERR_INVALID_ARG, "tr_trace_shadow_rays: null");
    if (!n) return TR_OK;
    DevBuf o, d, t, out;
    int32_t st = TR_OK;
    auto run = [&]() -> int32_t {
        TR_TRY(o.ensure((size_t)n * 12));
        TR_TRY(d.ensure((size_t)n * 12));
        TR_TRY(t.ensure((size_t)n * 4));
        TR_TRY(out.ensure(n));
        TR_CUDA(cudaMemcpyAsync(o.p, origins, (size_t)n * 12, cudaMemcpyHostToDevice, c->stream));
        TR_CUDA(cudaMemcpyAsync(d.p, directions, (size_t)n * 12, cudaMemcpyHostToDevice, c->stream));
        TR_CUDA(cudaMemcpyAsync(t.p, t_max, (size_t)n * 4, cudaMemcpyHostToDevice, c->stream));
        TR_TRY(launch_trace_rays(c, n, o.as<float>(), d.as<float>(), t.as<float>(), out.as<uint8_t>()));
        TR_CUDA(cudaMemcpyAsync(lit, out.p, n, cudaMemcpyDeviceToHost, c->stream));
        TR_CUDA(cudaStreamSynchronize(c->stream));
        return TR_OK;
    };
    st = run();
    cudaStreamSynchronize(c->stream);
    o.release(); d.release(); t.release(); out.release();
    return st;
}

int32_t tr_read_shadow_mask(tr_ctx* c, int32_t layer, uint32_t* mask) {
    TR_CHECK_CTX(c);
    if (layer < 0 || layer > 1 || !mask) return fail(TR_ERR_INVALID_ARG, "tr_read_shadow_mask: bad argument");
    const size_t plane = (size_t)c->width * c->height;
    if (c->shadow_mask[layer].bytes < plane * 20) return fail(TR_ERR_STATE, "tr_read_shadow_mask: layer %d was not shaded with ray queries", layer);
    // band rows only; the rest of the caller's buffer is left untouched
    for (int k = 0; k < 5; k++) {
        const size_t off = plane * k + (size_t)c->band_y0 * c->width;
        TR_CUDA(cudaMemcpyAsync(mask + off, c->shadow_mask[layer].as<uint32_t>() + off, (size_t)(c->band_y1 - c->band_y0) * c->width * 4,
                                cudaMemcpyDeviceToHost, c->stream));
    }
    TR_CUDA(cudaStreamSynchronize(c->stream));
    return TR_OK;
}

// ------------------------------------------------------------------ per-frame passes
int32_t tr_cull(tr_ctx* c, const tr_culling_push_constants* pc) {
    TR_CHECK_CTX(c);
    if (!pc) return fail(TR_ERR_INVALID_ARG, "tr_cull: null");
    pass_begin(c, P_CULL);
    TR_TRY(launch_cull(c, *pc));
    pass_end(c, P_CULL);
    return TR_OK;
}

int32_t tr_build_clusters(tr_ctx* c, const tr_write_cluster_data_push_constants* pc) {
    TR_CHECK_CTX(c);
    if (!pc) return fail(TR_ERR_INVALID_ARG, "tr_build_clusters: null");
    return launch_build_clusters(c, *pc);
}

int32_t tr_assign_lights(tr_ctx* c, const tr_assign_lights_push_constants* pc) {
    TR_CHECK_CTX(c);
    if (!pc) return fail(TR_ERR_INVALID_ARG, "tr_assign_lights: null");
    pass_begin(c, P_LIGHTS);
    TR_TRY(launch_assign_lights(c, *pc));
    pass_end(c, P_LIGHTS);
    return TR_OK;
}

int32_t tr_visibility(tr_ctx* c, const tr_push_constants* pc) {
    TR_CHECK_CTX(c);
    TR_TRY(check_pc(c, pc, "tr_visibility"));
    pass_begin(c, P_VIS);
    TR_TRY(launch_visibility(c, *pc));
    pass_end(c, P_VIS);
    return TR_OK;
}

int32_t tr_shade_opaque(tr_ctx* c, const tr_push_constants* pc) {
    TR_CHECK_CTX(c);
    TR_NOT_GROUPED(c, "tr_shade_opaque", "tr_group_frame");
    return shade_opaque(c, pc);
}

int32_t tr_allgather_opaque(tr_ctx* c) {
    TR_CHECK_CTX(c);
    TR_NOT_GROUPED(c, "tr_allgather_opaque", "tr_group_frame");
    if (c->n_ranks <= 1) return TR_OK;
    if (!c->opaque_valid) return fail(TR_ERR_STATE, "tr_allgather_opaque: no opaque frame");
    pass_begin(c, P_GATHER);
    TR_TRY(comm_allgather_opaque(c));
    pass_end(c, P_GATHER);
    return TR_OK;
}

int32_t tr_generate_mips(tr_ctx* c) {
    TR_CHECK_CTX(c);
    if (!c->opaque_valid) return fail(TR_ERR_STATE, "tr_generate_mips: no opaque frame (tr_shade_opaque / tr_set_opaque_frame)");
    pass_begin(c, P_MIPS);
    TR_TRY(launch_generate_mips(c->pyramid.as<uint2>(), c->levels, c->level_w, c->level_h, c->level_off,
                                c->mip_counter.as<uint32_t>(), c->sm_count, c->stream));
    pass_end(c, P_MIPS);
    c->mips_valid = true;
    return TR_OK;
}

int32_t tr_shade_transmission(tr_ctx* c, const tr_push_constants* pc) {
    TR_CHECK_CTX(c);
    ShadeLaunch s;
    TR_TRY(fill_shade(c, pc, TR_LAYER_TRANSMISSIVE, &s, "tr_shade_transmission"));
    if (!c->mips_valid) return fail(TR_ERR_STATE, "tr_shade_transmission: opaque pyramid not built (tr_generate_mips)");
    if (!c->lut_w) return fail(TR_ERR_STATE, "tr_shade_transmission: GGX LUT not set (tr_set_ggx_lut)");
    if (!c->hdr_valid) {  // LOAD of a target nothing rendered to: define it as zero
        TR_CUDA(cudaMemsetAsync(c->hdr.p, 0, (size_t)c->width * c->height * 8, c->stream));
        if (s.hdr_f32) TR_CUDA(cudaMemsetAsync(c->hdr_f32.p, 0, (size_t)c->width * c->height * 16, c->stream));
        c->hdr_valid = true;
    }
    pass_begin(c, P_TRANS);
    if (s.shadow_mask) {
        TR_TRY(launch_shadow_mask(s, c->sm_count, c->stream));
        TR_TRY(launch_shade_transmission_shadowed(s, c->sm_count, c->stream));
    } else {
        TR_TRY(launch_shade_transmission(s, c->sm_count, c->stream));
    }
    pass_end(c, P_TRANS);
    return TR_OK;
}

int32_t tr_tonemap(tr_ctx* c, const tr_baked_lottes_tonemapper_params* params) {
    TR_CHECK_CTX(c);
    if (!params) return fail(TR_ERR_INVALID_ARG, "tr_tonemap: null");
    if (!c->hdr_valid) return fail(TR_ERR_STATE, "tr_tonemap: nothing rendered");
    if (c->copy_pending) TR_CUDA(cudaStreamWaitEvent(c->stream, c->ev_copy_done, 0));  // the previous band is still being read back
    pass_begin(c, P_TONEMAP);
    TR_TRY(launch_tonemap(c->hdr.as<uint2>(), c->srgb8.as<uchar4>(), c->band_y0 * c->width, c->band_y1 * c->width, *params,
                          c->sm_count, c->stream));
    pass_end(c, P_TONEMAP);
    c->srgb_valid = true;
    return TR_OK;
}

int32_t tr_begin_frame(tr_ctx* c) {
    TR_CHECK_CTX(c);
    timing_next_frame(c);
    return TR_OK;
}

int32_t tr_frame(tr_ctx* c, const tr_frame_params* f) {
    TR_CHECK_CTX(c);
    TR_NOT_GROUPED(c, "tr_frame", "tr_group_frame");
    if (!f) return fail(TR_ERR_INVALID_ARG, "tr_frame: null");
    TR_TRY(frame_front(c, f));
    // peer-store path: a peer's opaque pass writes into THIS rank's mip 0, which the previous frame's transmissive
    // pass may still be sampling -> cross-GPU barrier before anybody starts shading
    if (c->n_ranks > 1 && c->peers_attached) TR_TRY(comm_barrier(c));
    TR_TRY(shade_opaque(c, &f->push_constants));
    if (c->n_ranks > 1) TR_TRY(tr_allgather_opaque(c));  // NCCL all-gather, or (peer path) the barrier that ends the exchange
    return frame_back(c, f, nullptr);
}

int32_t tr_enable_timing(tr_ctx* c, int32_t enable) {
    TR_CHECK_CTX(c);
    if (enable && !c->ev_begin) {
        c->ev_begin = new (std::nothrow) cudaEvent_t[kTimingRing][P_COUNT];
        c->ev_end = new (std::nothrow) cudaEvent_t[kTimingRing][P_COUNT];
        c->ev_used = new (std::nothrow) bool[kTimingRing][P_COUNT]();
        if (!c->ev_begin || !c->ev_end || !c->ev_used) return fail(TR_ERR_OOM, "tr_enable_timing: host allocation failed");
        for (int f = 0; f < kTimingRing; f++)
            for (int i = 0; i < P_COUNT; i++) {
                TR_CUDA(cudaEventCreate(&c->ev_begin[f][i]));
                TR_CUDA(cudaEventCreate(&c->ev_end[f][i]));
            }
    }
    c->timing = enable != 0;
    c->timing_first = c->timing_frame + 1;  // totals restart at the next tr_frame
    return TR_OK;
}

int32_t tr_read_frame_times(tr_ctx* c, tr_frame_times* out) {
    TR_CHECK_CTX(c);
    if (!out) return fail(TR_ERR_INVALID_ARG, "tr_read_frame_times: null");
    if (!c->ev_begin) return fail(TR_ERR_STATE, "tr_read_frame_times: timing was never enabled (tr_enable_timing)");
    TR_CUDA(cudaStreamSynchronize(c->stream));
    memset(out, 0, sizeof(*out));
    sum_frame_times(c, slot_of(c), out);
    return TR_OK;
}

int32_t tr_read_pass_totals(tr_ctx* c, tr_frame_times* sum, uint32_t* n_frames) {
    TR_CHECK_CTX(c);
    if (!sum || !n_frames) return fail(TR_ERR_INVALID_ARG, "tr_read_pass_totals: null");
    if (!c->ev_begin) return fail(TR_ERR_STATE, "tr_read_pass_totals: timing was never enabled (tr_enable_timing)");
    TR_CUDA(cudaStreamSynchronize(c->stream));
    memset(sum, 0, sizeof(*sum));
    uint32_t n = 0;
    for (uint64_t f = c->timing_first; f <= c->timing_frame; f++) n += (uint32_t)sum_frame_times(c, (int)(f % kTimingRing), sum);
    *n_frames = n;
    c->timing_first = c->timing_frame + 1;
    return TR_OK;
}

// ------------------------------------------------------------------ parity hooks
int32_t tr_set_gbuffer(tr_ctx* c, int32_t layer, const tr_gbuffer_planes* g) {
    TR_CHECK_CTX(c);
    if (layer < 0 || layer > 1 || !g || !g->depth || !g->normal || !g->material_id)
        return fail(TR_ERR_INVALID_ARG, "tr_set_gbuffer: bad layer or missing depth/normal/material_id plane");
    const size_t npx = (size_t)c->width * c->height;
    TR_TRY(ensure_layer(c, layer, g->position != nullptr));
    GLayer& L = c->layer[layer];
    TR_CUDA(cudaMemcpyAsync(L.depth.p, g->depth, npx * 4, cudaMemcpyHostToDevice, c->stream));
    TR_CUDA(cudaMemcpyAsync(L.normal.p, g->normal, npx * 12, cudaMemcpyHostToDevice, c->stream));
    if (g->uv) TR_CUDA(cudaMemcpyAsync(L.uv.p, g->uv, npx * 8, cudaMemcpyHostToDevice, c->stream));
    else TR_CUDA(cudaMemsetAsync(L.uv.p, 0, npx * 8, c->stream));
    TR_CUDA(cudaMemcpyAsync(L.material_id.p, g->material_id, npx * 4, cudaMemcpyHostToDevice, c->stream));
    if (g->scale) TR_CUDA(cudaMemcpyAsync(L.scale.p, g->scale, npx * 4, cudaMemcpyHostToDevice, c->stream));
    else {  // model_scale 1.0 everywhere
        std::vector<float> ones(npx, 1.0f);
        TR_CUDA(cudaMemcpyAsync(L.scale.p, ones.data(), npx * 4, cudaMemcpyHostToDevice, c->stream));  // ordered after a frame in flight
        TR_CUDA(cudaStreamSynchronize(c->stream));  // `ones` is a local
    }
    if (g->position) TR_CUDA(cudaMemcpyAsync(L.position.p, g->position, npx * 12, cudaMemcpyHostToDevice, c->stream));
    if (c->materials_textured) {
        if (g->duv) TR_CUDA(cudaMemcpyAsync(L.duv.p, g->duv, npx * 16, cudaMemcpyHostToDevice, c->stream));
        else TR_CUDA(cudaMemsetAsync(L.duv.p, 0, npx * 16, c->stream));
        if (g->ddepth) TR_CUDA(cudaMemcpyAsync(L.ddepth.p, g->ddepth, npx * 8, cudaMemcpyHostToDevice, c->stream));
        else TR_CUDA(cudaMemsetAsync(L.ddepth.p, 0, npx * 8, c->stream));
    }
    L.has_position = g->position != nullptr;
    L.valid = true;
    return TR_OK;
}

int32_t tr_read_gbuffer(tr_ctx* c, int32_t layer, const tr_gbuffer_planes_out* g) {
    TR_CHECK_CTX(c);
    if (layer < 0 || layer > 1 || !g) return fail(TR_ERR_INVALID_ARG, "tr_read_gbuffer: bad arguments");
    GLayer& L = c->layer[layer];
    if (!L.valid) return fail(TR_ERR_STATE, "tr_read_gbuffer: layer %d has no G-buffer", layer);
    const size_t npx = (size_t)c->width * c->height;
    TR_CUDA(cudaStreamSynchronize(c->stream));
    TR_TRY(check_device_status(c, "tr_read_gbuffer"));
    if (g->depth) TR_CUDA(cudaMemcpy(g->depth, L.depth.p, npx * 4, cudaMemcpyDeviceToHost));
    if (g->normal) TR_CUDA(cudaMemcpy(g->normal, L.normal.p, npx * 12, cudaMemcpyDeviceToHost));
    if (g->uv) TR_CUDA(cudaMemcpy(g->uv, L.uv.p, npx * 8, cudaMemcpyDeviceToHost));
    if (g->material_id) TR_CUDA(cudaMemcpy(g->material_id, L.material_id.p, npx * 4, cudaMemcpyDeviceToHost));
    if (g->scale) TR_CUDA(cudaMemcpy(g->scale, L.scale.p, npx * 4, cudaMemcpyDeviceToHost));
    if (g->position && L.has_position) TR_CUDA(cudaMemcpy(g->position, L.position.p, npx * 12, cudaMemcpyDeviceToHost));
    if (g->duv && L.duv.p) TR_CUDA(cudaMemcpy(g->duv, L.duv.p, npx * 16, cudaMemcpyDeviceToHost));
    if (g->ddepth && L.ddepth.p) TR_CUDA(cudaMemcpy(g->ddepth, L.ddepth.p, npx * 8, cudaMemcpyDeviceToHost));
    return TR_OK;
}

int32_t tr_set_opaque_frame(tr_ctx* c, const uint16_t* rgba16f) {
    TR_CHECK_CTX(c);
    if (!rgba16f) return fail(TR_ERR_INVALID_ARG, "tr_set_opaque_frame: null");
    TR_CUDA(cudaMemcpyAsync(c->pyramid.as<uint2>() + c->level_off[0], rgba16f, (size_t)c->width * c->height * 8,
                            cudaMemcpyHostToDevice, c->stream));
    c->opaque_valid = true;
    c->mips_valid = false;
    return TR_OK;
}

int32_t tr_set_hdr(tr_ctx* c, const uint16_t* rgba16f) {
    TR_CHECK_CTX(c);
    if (!rgba16f) return fail(TR_ERR_INVALID_ARG, "tr_set_hdr: null");
    TR_CUDA(cudaMemcpyAsync(c->hdr.p, rgba16f, (size_t)c->width * c->height * 8, cudaMemcpyHostToDevice, c->stream));
    c->hdr_valid = true;
    return TR_OK;
}

int32_t tr_set_cluster_lights(tr_ctx* c, const uint32_t* counts, const uint32_t* indices) {
    TR_CHECK_CTX(c);
    if (!c->have_uniforms) return fail(TR_ERR_STATE, "tr_set_cluster_lights: uniforms not set");
    if (!counts || !indices) return fail(TR_ERR_INVALID_ARG, "tr_set_cluster_lights: null");
    for (uint32_t k = 0; k < c->n_clusters; k++) {
        if (counts[k] > TR_MAX_LIGHTS_PER_CLUSTER)
            return fail(TR_ERR_INVALID_ARG, "tr_set_cluster_lights: cluster %u lists %u lights (at most %u)", k, counts[k], TR_MAX_LIGHTS_PER_CLUSTER);
        for (uint32_t i = 0; i < counts[k]; i++)
            if (indices[(size_t)k * TR_MAX_LIGHTS_PER_CLUSTER + i] >= c->n_lights)
                return fail(TR_ERR_INVALID_ARG, "tr_set_cluster_lights: cluster %u names light %u of %u", k,
                            indices[(size_t)k * TR_MAX_LIGHTS_PER_CLUSTER + i], c->n_lights);
    }
    TR_TRY(upload(c, c->cluster_counts, counts, (size_t)c->n_clusters * 4));
    TR_TRY(upload(c, c->cluster_indices, indices, (size_t)c->n_clusters * TR_MAX_LIGHTS_PER_CLUSTER * 4));
    c->cluster_lights_valid = true;
    return TR_OK;
}

int32_t tr_read_visible_instances(tr_ctx* c, uint32_t* ids, uint32_t capacity, uint32_t* n_visible) {
    TR_CHECK_CTX(c);
    if (!c->cull_valid) return fail(TR_ERR_STATE, "tr_read_visible_instances: tr_cull has not run");
    TR_CUDA(cudaStreamSynchronize(c->stream));
    uint32_t n = 0;
    TR_CUDA(cudaMemcpy(&n, c->d_cull_scalars, 4, cudaMemcpyDeviceToHost));
    if (n_visible) *n_visible = n;
    if (ids) {
        if (capacity < n) return fail(TR_ERR_INVALID_ARG, "tr_read_visible_instances: capacity %u < %u", capacity, n);
        TR_CUDA(cudaMemcpy(ids, c->visible_ids.p, (size_t)n * 4, cudaMemcpyDeviceToHost));
    }
    return TR_OK;
}

int32_t tr_read_instance_counts(tr_ctx* c, uint32_t* counts, uint32_t capacity) {
    TR_CHECK_CTX(c);
    if (!c->cull_valid) return fail(TR_ERR_STATE, "tr_read_instance_counts: tr_cull has not run");
    if (!counts || capacity < c->n_primitives) return fail(TR_ERR_INVALID_ARG, "tr_read_instance_counts: capacity");
    TR_CUDA(cudaStreamSynchronize(c->stream));
    TR_CUDA(cudaMemcpy(counts, c->d_instance_counts, (size_t)c->n_primitives * 4, cudaMemcpyDeviceToHost));
    return TR_OK;
}

int32_t tr_read_draws(tr_ctx* c, uint32_t bucket, tr_draw_indexed_indirect_command* cmds, uint32_t capacity, uint32_t* n_draws) {
    TR_CHECK_CTX(c);
    if (!c->cull_valid) return fail(TR_ERR_STATE, "tr_read_draws: tr_cull has not run");
    if (bucket >= TR_NUM_DRAW_BUFFERS) return fail(TR_ERR_INVALID_ARG, "tr_read_draws: bucket %u", bucket);
    TR_CUDA(cudaStreamSynchronize(c->stream));
    uint32_t n = 0;
    TR_CUDA(cudaMemcpy(&n, c->d_cull_scalars + 2 + bucket, 4, cudaMemcpyDeviceToHost));
    if (n_draws) *n_draws = n;
    if (cmds) {
        if (capacity < n) return fail(TR_ERR_INVALID_ARG, "tr_read_draws: capacity %u < %u", capacity, n);
        TR_CUDA(cudaMemcpy(cmds, c->draws[bucket].p, (size_t)n * sizeof(tr_draw_indexed_indirect_command), cudaMemcpyDeviceToHost));
    }
    return TR_OK;
}

int32_t tr_read_cluster_aabbs(tr_ctx* c, tr_cluster_aabb* aabbs, uint32_t capacity) {
    TR_CHECK_CTX(c);
    if (!c->clusters_valid) return fail(TR_ERR_STATE, "tr_read_cluster_aabbs: tr_build_clusters has not run");
    if (!aabbs || capacity < c->n_clusters) return fail(TR_ERR_INVALID_ARG, "tr_read_cluster_aabbs: capacity");
    TR_CUDA(cudaStreamSynchronize(c->stream));
    TR_CUDA(cudaMemcpy(aabbs, c->cluster_aabbs.p, (size_t)c->n_clusters * sizeof(tr_cluster_aabb), cudaMemcpyDeviceToHost));
    return TR_OK;
}

int32_t tr_read_cluster_lights(tr_ctx* c, uint32_t* counts, uint32_t* indices) {
    TR_CHECK_CTX(c);
    if (!c->cluster_lights_valid) return fail(TR_ERR_STATE, "tr_read_cluster_lights: no light lists");
    TR_CUDA(cudaStreamSynchronize(c->stream));
    if (counts) TR_CUDA(cudaMemcpy(counts, c->cluster_counts.p, (size_t)c->n_clusters * 4, cudaMemcpyDeviceToHost));
    if (indices) TR_CUDA(cudaMemcpy(indices, c->cluster_indices.p, (size_t)c->n_clusters * TR_MAX_LIGHTS_PER_CLUSTER * 4, cudaMemcpyDeviceToHost));
    return TR_OK;
}

int32_t tr_read_hdr(tr_ctx* c, uint16_t* rgba16f) {
    TR_CHECK_CTX(c);
    if (!rgba16f) return fail(TR_ERR_INVALID_ARG, "tr_read_hdr: null");
    if (!c->hdr_valid) return fail(TR_ERR_STATE, "tr_read_hdr: nothing rendered");
    TR_CUDA(cudaStreamSynchronize(c->stream));
    TR_CUDA(cudaMemcpy(rgba16f, c->hdr.p, (size_t)c->width * c->height * 8, cudaMemcpyDeviceToHost));
    return check_device_status(c, "tr_read_hdr");
}

int32_t tr_read_hdr_f32(tr_ctx* c, float* rgba32f) {
    TR_CHECK_CTX(c);
    if (!rgba32f) return fail(TR_ERR_INVALID_ARG, "tr_read_hdr_f32: null");
    if (!(c->flags & TR_FLAG_HDR_F32_DEBUG)) return fail(TR_ERR_STATE, "tr_read_hdr_f32: context created without TR_FLAG_HDR_F32_DEBUG");
    if (!c->hdr_valid) return fail(TR_ERR_STATE, "tr_read_hdr_f32: nothing rendered");
    TR_CUDA(cudaStreamSynchronize(c->stream));
    TR_CUDA(cudaMemcpy(rgba32f, c->hdr_f32.p, (size_t)c->width * c->height * 16, cudaMemcpyDeviceToHost));
    return check_device_status(c, "tr_read_hdr_f32");
}

int32_t tr_read_pyramid_level(tr_ctx* c, uint32_t level, uint16_t* rgba16f, uint32_t* w, uint32_t* h) {
    TR_CHECK_CTX(c);
    if (level >= c->levels) return fail(TR_ERR_INVALID_ARG, "tr_read_pyramid_level: level %u of %u", level, c->levels);
    if (level == 0 ? !c->opaque_valid : !c->mips_valid) return fail(TR_ERR_STATE, "tr_read_pyramid_level: level not built");
    if (w) *w = c->level_w[level];
    if (h) *h = c->level_h[level];
    if (rgba16f) {
        TR_CUDA(cudaStreamSynchronize(c->stream));
        TR_CUDA(cudaMemcpy(rgba16f, c->pyramid.as<uint2>() + c->level_off[level], (size_t)c->level_w[level] * c->level_h[level] * 8,
                           cudaMemcpyDeviceToHost));
    }
    return TR_OK;
}

int32_t tr_read_srgb8(tr_ctx* c, uint8_t* rgba8) {
    TR_CHECK_CTX(c);
    if (!rgba8) return fail(TR_ERR_INVALID_ARG, "tr_read_srgb8: null");
    if (!c->srgb_valid) return fail(TR_ERR_STATE, "tr_read_srgb8: tr_tonemap has not run");
    const size_t off = (size_t)c->band_y0 * c->width * 4, bytes = (size_t)(c->band_y1 - c->band_y0) * c->width * 4;
    TR_CUDA(cudaMemcpyAsync(rgba8 + off, c->srgb8.as<uint8_t>() + off, bytes, cudaMemcpyDeviceToHost, c->stream));
    TR_CUDA(cudaStreamSynchronize(c->stream));
    return check_device_status(c, "tr_read_srgb8");
}

int32_t tr_read_srgb8_async(tr_ctx* c, uint8_t* rgba8) {
    TR_CHECK_CTX(c);
    if (!rgba8) return fail(TR_ERR_INVALID_ARG, "tr_read_srgb8_async: null");
    if (!c->srgb_valid) return fail(TR_ERR_STATE, "tr_read_srgb8_async: tr_tonemap has not run");
    if (!c->copy_stream) {
        TR_CUDA(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
        TR_CUDA(cudaEventCreateWithFlags(&c->ev_frame_done, cudaEventDisableTiming));
        TR_CUDA(cudaEventCreateWithFlags(&c->ev_copy_done, cudaEventDisableTiming));
    }
    const size_t off = (size_t)c->band_y0 * c->width * 4, bytes = (size_t)(c->band_y1 - c->band_y0) * c->width * 4;
    TR_CUDA(cudaEventRecord(c->ev_frame_done, c->stream));
    TR_CUDA(cudaStreamWaitEvent(c->copy_stream, c->ev_frame_done, 0));
    TR_CUDA(cudaMemcpyAsync(rgba8 + off, c->srgb8.as<uint8_t>() + off, bytes, cudaMemcpyDeviceToHost, c->copy_stream));
    TR_CUDA(cudaEventRecord(c->ev_copy_done, c->copy_stream));
    c->copy_pending = true;
    return TR_OK;
}

int32_t tr_wait_readback(tr_ctx* c) {
    TR_CHECK_CTX(c);
    if (c->copy_pending) TR_CUDA(cudaEventSynchronize(c->ev_copy_done));
    return check_device_status(c, "tr_wait_readback");  // an overflowed visibility pass must not pass for a good frame
}

int32_t tr_read_texture_level(tr_ctx* c, uint32_t index, uint32_t level, float* rgba32f, uint32_t* w, uint32_t* h) {
    TR_CHECK_CTX(c);
    if (index >= TR_MAX_IMAGES) return fail(TR_ERR_INVALID_ARG, "tr_read_texture_level: image %u of at most %u", index, TR_MAX_IMAGES);
    const trd::TexDesc& d = c->h_tex[index];
    if (!d.base) return fail(TR_ERR_STATE, "tr_read_texture_level: image %u is not bound", index);
    if (level >= d.levels) return fail(TR_ERR_INVALID_ARG, "tr_read_texture_level: level %u of %u", level, d.levels);
    const uint32_t lw = d.w >> level ? d.w >> level : 1u, lh = d.h >> level ? d.h >> level : 1u;
    if (w) *w = lw;
    if (h) *h = lh;
    if (rgba32f) {
        TR_CUDA(cudaMemcpyAsync(rgba32f, d.base + d.off[level], (size_t)lw * lh * 16, cudaMemcpyDeviceToHost, c->stream));
        TR_CUDA(cudaStreamSynchronize(c->stream));
    }
    return TR_OK;
}

int32_t tr_mip_levels(tr_ctx* c, uint32_t* levels) {
    if (!c || !levels) return fail(TR_ERR_INVALID_ARG, "tr_mip_levels: null");
    *levels = c->levels;
    return TR_OK;
}

}  // extern "C"

// ------------------------------------------------------------------ glam-pbr contract batch evaluators
template <typename In, typename Out, typename F>
static int32_t eval_batch(tr_ctx* c, uint32_t n, const In* in, Out* out, F launch) {
    if (n == 0) return TR_OK;
    if (!in || !out) return fail(TR_ERR_INVALID_ARG, "tr_eval_*: null");
    DevBuf din, dout;
    int32_t s = din.ensure((size_t)n * sizeof(In));
    if (s == TR_OK) s = dout.ensure((size_t)n * sizeof(Out));
    if (s == TR_OK && cudaMemcpyAsync(din.p, in, (size_t)n * sizeof(In), cudaMemcpyHostToDevice, c->stream) != cudaSuccess)
        s = fail(TR_ERR_CUDA, "tr_eval_*: upload failed");
    if (s == TR_OK) s = launch(din.as<In>(), dout.as<Out>());
    if (s == TR_OK && cudaMemcpyAsync(out, dout.p, (size_t)n * sizeof(Out), cudaMemcpyDeviceToHost, c->stream) != cudaSuccess)
        s = fail(TR_ERR_CUDA, "tr_eval_*: download failed");
    cudaError_t e = cudaStreamSynchronize(c->stream);
    if (s == TR_OK && e != cudaSuccess) s = fail(TR_ERR_CUDA, "tr_eval_*: %s", cudaGetErrorString(e));
    din.release();
    dout.release();
    return s;
}

extern "C" {

int32_t tr_eval_basic_brdf(tr_ctx* c, uint32_t n, const tr_basic_brdf_params* params, tr_brdf_result* out) {
    TR_CHECK_CTX(c);
    return eval_batch(c, n, params, out, [&](const tr_basic_brdf_params* i, tr_brdf_result* o) {
        return launch_eval_basic_brdf(n, i, o, c->stream);
    });
}

int32_t tr_eval_transmission_btdf(tr_ctx* c, uint32_t n, const tr_transmission_btdf_params* params, tr_vec3* out) {
    TR_CHECK_CTX(c);
    return eval_batch(c, n, params, out, [&](const tr_transmission_btdf_params* i, tr_vec3* o) {
        return launch_eval_transmission_btdf(n, i, o, c->stream);
    });
}

int32_t tr_eval_point_light(tr_ctx* c, uint32_t n, const tr_point_light_params* params, tr_point_light_result* out) {
    TR_CHECK_CTX(c);
    return eval_batch(c, n, params, out, [&](const tr_point_light_params* i, tr_point_light_result* o) {
        return launch_eval_point_light(n, i, o, c->stream);
    });
}

int32_t tr_eval_ibl_volume_refraction(tr_ctx* c, uint32_t n, const tr_mat4* proj_view,
                                      const tr_ibl_volume_refraction_params* params, tr_vec3* out) {
    TR_CHECK_CTX(c);
    if (!proj_view) return fail(TR_ERR_INVALID_ARG, "tr_eval_ibl_volume_refraction: null proj_view");
    if (!c->mips_valid) return fail(TR_ERR_STATE, "tr_eval_ibl_volume_refraction: opaque pyramid not built");
    if (!c->lut_w) return fail(TR_ERR_STATE, "tr_eval_ibl_volume_refraction: GGX LUT not set");
    trd::mat4 pv;
    memcpy(&pv, proj_view, sizeof(pv));
    const trd::PyramidDesc pyr = pyramid_desc(c);
    const trd::LutDesc lut = lut_desc(c);
    return eval_batch(c, n, params, out, [&](const tr_ibl_volume_refraction_params* i, tr_vec3* o) {
        return launch_eval_ibl(n, pv, i, o, pyr, lut, c->stream);
    });
}

int32_t tr_raster_stats(tr_ctx* c, uint64_t out[4], int32_t reset) {
    TR_CHECK_CTX(c);
    if (!out) return fail(TR_ERR_INVALID_ARG, "tr_raster_stats: null");
    memset(out, 0, 32);
    if (!c->dev_status.p) return TR_OK;
    TR_CUDA(cudaStreamSynchronize(c->stream));
    TR_CUDA(cudaMemcpy(out, c->dev_status.as<unsigned char>() + 16, 32, cudaMemcpyDeviceToHost));
    if (reset) TR_CUDA(cudaMemset(c->dev_status.as<unsigned char>() + 16, 0, 32));
    return TR_OK;
}

int32_t tr_launch_count(uint64_t* out) {
    if (!out) return fail(TR_ERR_INVALID_ARG, "tr_launch_count: null");
    *out = tr::g_launches.load();
    return TR_OK;
}

int32_t tr_device_buffer(tr_ctx* c, int32_t what, void** device_ptr, size_t* bytes) {
    if (!c || !device_ptr) return fail(TR_ERR_INVALID_ARG, "tr_device_buffer: null");
    const size_t npx = (size_t)c->width * c->height;
    switch (what) {
        case TR_BUF_OPAQUE_MIP0: *device_ptr = c->pyramid.as<uint2>() + c->level_off[0]; if (bytes) *bytes = npx * 8; break;
        case TR_BUF_HDR: *device_ptr = c->hdr.p; if (bytes) *bytes = npx * 8; break;
        case TR_BUF_SRGB8: *device_ptr = c->srgb8.p; if (bytes) *bytes = npx * 4; break;
        case TR_BUF_HDR_F32:
            if (!(c->flags & TR_FLAG_HDR_F32_DEBUG)) return fail(TR_ERR_STATE, "tr_device_buffer: no fp32 HDR target");
            *device_ptr = c->hdr_f32.p; if (bytes) *bytes = npx * 16; break;
        default: return fail(TR_ERR_INVALID_ARG, "tr_device_buffer: unknown buffer %d", what);
    }
    return TR_OK;
}

}  // extern "C"
