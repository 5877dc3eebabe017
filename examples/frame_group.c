/* examples/frame_group.c — one frame across several contexts from one host thread (tr_group_*), in plain C.
 *
 *   gcc -std=c11 -I include examples/frame_group.c -L transmission_renderer_b200 -ltr -Wl,-rpath,$PWD/transmission_renderer_b200 -lm -o frame_group
 *
 * The reference's host is one thread with one queue (src/main.rs:243, 1290-1294).  This host makes one context per visible
 * device (two on device 0 when there is only one), joins them into a group, which gives member k the k-th band of the frame,
 * and renders the frame of examples/frame.c through tr_group_frame.  The scene is uploaded to member 0 only, and
 * tr_group_replicate_scene copies it into the other members GPU to GPU, in stream order (uploading to every member, as to
 * single contexts, works too).  There is no CPU fallback: without a CUDA device tr_create fails and the program says so and exits with
 * status 3.
 */
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "tr_abi.h"

#define MAX_MEMBERS 8

#define CHECK(call)                                                               \
    do {                                                                          \
        int32_t st_ = (call);                                                     \
        if (st_ != TR_OK) {                                                       \
            fprintf(stderr, "%s -> %d: %s\n", #call, st_, tr_last_error());       \
            return 3;                                                             \
        }                                                                         \
    } while (0)

static void identity(tr_mat4* m) {
    memset(m, 0, sizeof(*m));
    m->col[0].x = m->col[1].y = m->col[2].z = m->col[3].w = 1.0f;
}

/* the scene of examples/frame.c: one triangle in clip space, one material, no point lights */
static int upload_scene(tr_ctx* ctx, uint32_t w, uint32_t h) {
    const float pos[9] = {-0.8f, -0.8f, 0.5f, 0.8f, -0.8f, 0.5f, 0.0f, 0.8f, 0.5f};
    const float nrm[9] = {0, 0, 1, 0, 0, 1, 0, 0, 1};
    const float uv[6] = {0, 0, 1, 0, 0.5f, 1};
    const uint32_t idx[6] = {0, 1, 2, 0, 2, 1};
    tr_primitive_info prim;
    memset(&prim, 0, sizeof(prim));
    prim.packed_bounding_sphere.w = 2.0f;
    prim.index_count = 6;
    tr_instance inst;
    memset(&inst, 0, sizeof(inst));
    inst.transform.translation_and_scale.w = 1.0f;
    inst.transform.rotation.w = 1.0f;
    tr_material_info mat;
    memset(&mat, 0, sizeof(mat));
    mat.textures.diffuse = mat.textures.metallic_roughness = mat.textures.normal_map = mat.textures.emissive = -1;
    mat.textures.occlusion = mat.textures.transmission = mat.textures.thickness = mat.textures.specular = mat.textures.specular_colour = -1;
    mat.roughness_factor = 0.5f;
    mat.alpha_clipping_cutoff = 0.5f;
    mat.diffuse_factor.x = 0.8f; mat.diffuse_factor.y = 0.3f; mat.diffuse_factor.z = 0.2f; mat.diffuse_factor.w = 1.0f;
    mat.index_of_refraction = 1.5f;
    mat.attenuation_distance = INFINITY;
    mat.specular_factor = 1.0f;
    mat.specular_colour_factor.x = mat.specular_colour_factor.y = mat.specular_colour_factor.z = 1.0f;
    tr_uniforms u;
    memset(&u, 0, sizeof(u));
    u.light_clustering_coefficients.z_near = 0.01f;
    u.light_clustering_coefficients.z_far = 500.0f;
    u.light_clustering_coefficients.num_depth_slices = 24;
    u.light_clustering_coefficients.scale = 24.0f / log2f(500.0f / 0.01f);
    u.light_clustering_coefficients.bias = -(24.0f * log2f(0.01f) / log2f(500.0f / 0.01f));
    u.sun_dir.z = 1.0f;
    u.sun_intensity.x = u.sun_intensity.y = u.sun_intensity.z = 3.0f;
    u.num_clusters.x = 12; u.num_clusters.y = 8;
    u.cluster_size_in_pixels.x = (float)w / 12.0f; u.cluster_size_in_pixels.y = (float)h / 8.0f;

    CHECK(tr_set_mesh(ctx, pos, nrm, uv, 3, idx, 6));
    CHECK(tr_set_primitives(ctx, &prim, 1));
    CHECK(tr_set_instances(ctx, &inst, 1));
    CHECK(tr_set_materials(ctx, &mat, 1));
    CHECK(tr_set_lights(ctx, NULL, 0));
    CHECK(tr_set_uniforms(ctx, &u));
    uint8_t lut[4 * 4 * 4];
    for (int i = 0; i < 16; i++) { lut[i * 4] = 128; lut[i * 4 + 1] = 32; lut[i * 4 + 2] = 0; lut[i * 4 + 3] = 255; }
    CHECK(tr_set_ggx_lut(ctx, lut, 4, 4));
    tr_write_cluster_data_push_constants wc;
    identity(&wc.inverse_perspective);
    wc.screen_dimensions.x = w; wc.screen_dimensions.y = h;
    CHECK(tr_build_clusters(ctx, &wc));
    return 0;
}

int main(int argc, char** argv) {
    const uint32_t w = 256, h = 144;
    /* devices: the command line (e.g. `frame_group 0 0 0 0`), else one per visible device, probed by creating contexts */
    tr_ctx* ctx[MAX_MEMBERS] = {0};
    uint32_t n = 0;
    printf("%s\n", tr_version());
    if (argc > 1) {
        for (int i = 1; i < argc && n < MAX_MEMBERS; i++) {
            tr_config cfg = {w, h, atoi(argv[i]), 0, 0, 0};
            CHECK(tr_create(&cfg, &ctx[n]));
            n++;
        }
    } else {
        tr_config cfg = {w, h, 0, 0, 0, 0};
        CHECK(tr_create(&cfg, &ctx[n]));   /* device 0, or the loud failure without a device */
        n++;
        for (int d = 1; n < MAX_MEMBERS; d++) {
            cfg.device = d;
            if (tr_create(&cfg, &ctx[n]) != TR_OK) break;   /* past the last device */
            n++;
        }
        if (n == 1) {   /* one device: two contexts on it run the same code two GPUs would */
            cfg.device = 0;
            CHECK(tr_create(&cfg, &ctx[n]));
            n++;
        }
    }
    tr_group* group = NULL;
    CHECK(tr_group_create(ctx, n, &group));
    if (upload_scene(ctx[0], w, h)) return 3;
    CHECK(tr_group_replicate_scene(group, 0, NULL));   /* no acceleration structures: no handles to collect */

    tr_frame_params f[MAX_MEMBERS];
    memset(f, 0, sizeof(f));
    for (uint32_t k = 0; k < n; k++) {   /* the same camera for every member; no ray queries, so no per-member handle */
        identity(&f[k].culling.view);
        f[k].culling.frustum_x_xz.x = 1.0f; f[k].culling.frustum_x_xz.y = 1.0f;
        f[k].culling.frustum_y_yz.x = 1.0f; f[k].culling.frustum_y_yz.y = 1.0f;
        identity(&f[k].assign_lights.view_matrix);
        f[k].assign_lights.view_rotation.w = 1.0f;
        identity(&f[k].push_constants.proj_view);
        f[k].push_constants.view_position.z = 5.0f;
        f[k].push_constants.framebuffer_size.x = w; f[k].push_constants.framebuffer_size.y = h;
        f[k].tonemap.a = 1.6f; f[k].tonemap.d = 0.977f; f[k].tonemap.b = 1.0f; f[k].tonemap.c = 1.0f; f[k].tonemap.saturation = 1.0f;
    }
    CHECK(tr_group_frame(group, f));

    uint8_t* rgba = (uint8_t*)malloc((size_t)w * h * 4);
    CHECK(tr_group_read_srgb8(group, rgba));
    unsigned long covered = 0;
    for (uint32_t i = 0; i < w * h; i++) covered += (rgba[i * 4] | rgba[i * 4 + 1] | rgba[i * 4 + 2]) != 0;
    printf("frame %ux%u over %u contexts: %lu lit pixels\n", w, h, n, covered);
    free(rgba);
    CHECK(tr_group_destroy(group));
    for (uint32_t k = 0; k < n; k++) CHECK(tr_destroy(ctx[k]));
    return 0;
}
