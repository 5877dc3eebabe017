// tr_host.hpp — the host side above the C ABI in C++ (header-only, C++17).
//
// The reference's host is compiled code (Rust, src/main.rs); there is no Rust toolchain in this environment, so the
// compiled-language mirror of what that host does for the path lives here, with the reference's names and argument
// meaning, on top of include/tr_abi.h (INTEGRATION.md shows the Rust binding of the same ABI):
//
//   * the per-frame inputs the reference computes on the CPU before it records a frame —
//       perspective_matrix_reversed            src/main.rs:39-54
//       Z_NEAR .. NUM_CLUSTERS                 src/main.rs:56-63
//       look_at_rh / yaw_pitch_camera          dolly YawPitch rig + glam Mat4::look_at_rh, src/main.rs:514-526
//       Sun::as_normal                         src/main.rs:2715-2722 (defaults :531-534)
//       LightClusterCoefficients::new          shared-structs/src/lib.rs:44-52
//       uniforms                               src/main.rs:536-552
//       culling / write_cluster_data / assign_lights push constants   src/main.rs:1728-1746, 1502-1505, 1785-1788
//       Light::new_point / new_spot            shared-structs/src/lib.rs:94-123
//       mip_levels_for_size, dispatch_count    src/main.rs:2590-2592, 2639-2641
//   * Renderer: an owning handle of a tr_ctx whose methods return through exceptions, the way every fallible function
//     of the reference returns anyhow::Result and is propagated with `?` (src/main.rs:93); record() (src/main.rs:1551) is
//     Renderer::frame.
//   * RendererGroup: several Renderers of one thread rendering the bands of one frame (tr_group_*), on one or more GPUs.
//
// tests/test_host_mirror.py compiles tests/host_mirror_dump.cpp against this header and compares every struct it builds
// with the Python restatement (transmission_renderer_b200/host.py) the parity tests use: identical bytes wherever no
// libm transcendental is involved, within 2 ulp where one is.  Nothing here touches the GPU except through tr_abi.h; a
// missing device or library fails in tr_create and surfaces as tr::Error — there is no CPU path.
#ifndef TR_HOST_HPP
#define TR_HOST_HPP

#include <cmath>
#include <cstdint>
#include <cstring>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "tr_abi.h"

namespace tr {

constexpr float Z_NEAR = 0.01f;            // src/main.rs:56
constexpr float Z_FAR = 500.0f;            // src/main.rs:57
constexpr uint32_t NUM_CLUSTERS_X = 24;    // src/main.rs:60
constexpr uint32_t NUM_CLUSTERS_Y = 16;    // src/main.rs:61
constexpr uint32_t NUM_DEPTH_SLICES = 16;  // src/main.rs:62
constexpr uint32_t NUM_CLUSTERS = NUM_CLUSTERS_X * NUM_CLUSTERS_Y * NUM_DEPTH_SLICES;

struct Vec3 {
    float x, y, z;
};
struct Quat {
    float x, y, z, w;
};
// row-major storage, m[row][col], math convention (a column vector is multiplied from the right); to_abi() transposes into
// glam's column-major Mat4
struct Mat4 {
    float m[4][4];
    static Mat4 zero() {
        Mat4 r;
        std::memset(&r, 0, sizeof r);
        return r;
    }
    static Mat4 identity() {
        Mat4 r = zero();
        for (int i = 0; i < 4; i++) r.m[i][i] = 1.0f;
        return r;
    }
    tr_mat4 to_abi() const {
        tr_mat4 o;
        for (int c = 0; c < 4; c++) {
            o.col[c].x = m[0][c];
            o.col[c].y = m[1][c];
            o.col[c].z = m[2][c];
            o.col[c].w = m[3][c];
        }
        return o;
    }
};

inline Mat4 mul(const Mat4& a, const Mat4& b) {   // fp32, sum over k in ascending order
    Mat4 r = Mat4::zero();
    for (int i = 0; i < 4; i++)
        for (int j = 0; j < 4; j++) {
            float s = 0.0f;
            for (int k = 0; k < 4; k++) s += a.m[i][k] * b.m[k][j];
            r.m[i][j] = s;
        }
    return r;
}

inline float dot(Vec3 a, Vec3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
inline Vec3 cross(Vec3 a, Vec3 b) { return {a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x}; }
inline Vec3 sub(Vec3 a, Vec3 b) { return {a.x - b.x, a.y - b.y, a.z - b.z}; }
inline Vec3 add(Vec3 a, Vec3 b) { return {a.x + b.x, a.y + b.y, a.z + b.z}; }
inline Vec3 normalize(Vec3 v) {   // glam: v * (1 / length)
    const float inv = 1.0f / std::sqrt(dot(v, v));
    return {v.x * inv, v.y * inv, v.z * inv};
}

// src/main.rs:39-54
inline Mat4 perspective_matrix_reversed(uint32_t width, uint32_t height) {
    const float aspect_ratio = (float)width / (float)height;
    const float vertical_fov = (float)(59.0 * 3.14159265358979323846 / 180.0);
    const float focal_length = 1.0f / (float)std::tan((double)(vertical_fov / 2.0f));
    const float a = Z_NEAR / (Z_FAR - Z_NEAR);
    const float b = Z_FAR * a;
    Mat4 r = Mat4::zero();
    r.m[0][0] = focal_length / aspect_ratio;
    r.m[1][1] = -focal_length;
    r.m[2][2] = a;
    r.m[3][2] = -1.0f;
    r.m[2][3] = b;
    return r;
}

// glam::Mat4::look_at_rh (src/main.rs:520-526)
inline Mat4 look_at_rh(Vec3 eye, Vec3 center, Vec3 up) {
    const Vec3 f = normalize(sub(center, eye));
    const Vec3 s = normalize(cross(f, up));
    const Vec3 u = cross(s, f);
    Mat4 r = Mat4::identity();
    r.m[0][0] = s.x; r.m[0][1] = s.y; r.m[0][2] = s.z;
    r.m[1][0] = u.x; r.m[1][1] = u.y; r.m[1][2] = u.z;
    r.m[2][0] = -f.x; r.m[2][1] = -f.y; r.m[2][2] = -f.z;
    r.m[0][3] = -dot(s, eye);
    r.m[1][3] = -dot(u, eye);
    r.m[2][3] = dot(f, eye);
    return r;
}

inline Vec3 rotate(Quat q, Vec3 v) {   // in double, rounded once
    const double bx = q.x, by = q.y, bz = q.z, w = q.w, vx = v.x, vy = v.y, vz = v.z;
    const double bb = bx * bx + by * by + bz * bz, vb = vx * bx + vy * by + vz * bz;
    const double cx = by * vz - bz * vy, cy = bz * vx - bx * vz, cz = bx * vy - by * vx;
    return {(float)(vx * (w * w - bb) + bx * (2.0 * vb) + cx * (2.0 * w)), (float)(vy * (w * w - bb) + by * (2.0 * vb) + cy * (2.0 * w)),
            (float)(vz * (w * w - bb) + bz * (2.0 * vb) + cz * (2.0 * w))};
}
inline Quat inverse(Quat q) { return {-q.x, -q.y, -q.z, q.w}; }

// The dolly YawPitch rig of src/main.rs:514-526: rotation = from_euler(YXZ, yaw, pitch, 0), view = look_at_rh(position,
// position + rotation * -Z, rotation * Y)
struct Camera {
    Mat4 view;
    Quat rotation;
    Vec3 position;
};
inline Camera yaw_pitch_camera(Vec3 position, double yaw_deg, double pitch_deg) {
    const double yaw = yaw_deg * 3.14159265358979323846 / 180.0, pitch = pitch_deg * 3.14159265358979323846 / 180.0;
    const double cy = std::cos(yaw / 2), sy = std::sin(yaw / 2), cp = std::cos(pitch / 2), sp = std::sin(pitch / 2);
    Camera c;
    c.rotation = {(float)(cy * sp), (float)(sy * cp), (float)(-sy * sp), (float)(cy * cp)};   // q_y(yaw) * q_x(pitch)
    c.position = position;
    c.view = look_at_rh(position, add(position, rotate(c.rotation, {0.0f, 0.0f, -1.0f})), rotate(c.rotation, {0.0f, 1.0f, 0.0f}));
    return c;
}

// Sun::as_normal, src/main.rs:2715-2722 (defaults :531-534)
inline Vec3 sun_as_normal(float pitch = 1.1f, float yaw = 4.8f) {
    return {std::cos(pitch) * std::sin(yaw), std::sin(pitch), std::cos(pitch) * std::cos(yaw)};
}

// LightClusterCoefficients::new, shared-structs/src/lib.rs:44-52
inline tr_light_cluster_coefficients light_cluster_coefficients(float z_near = Z_NEAR, float z_far = Z_FAR, uint32_t slices = NUM_DEPTH_SLICES) {
    const float l = std::log2(z_far / z_near);
    tr_light_cluster_coefficients c;
    c.z_near = z_near;
    c.z_far = z_far;
    c.scale = (float)slices / l;
    c.bias = -((float)slices * std::log2(z_near) / l);
    c.num_depth_slices = slices;
    return c;
}

// src/main.rs:536-552
inline tr_uniforms make_uniforms(uint32_t width, uint32_t height, Vec3 sun_dir = sun_as_normal(), Vec3 sun_intensity = {3.0f, 3.0f, 3.0f}) {
    tr_uniforms u;
    std::memset(&u, 0, sizeof u);
    u.light_clustering_coefficients = light_cluster_coefficients();
    u.sun_dir.x = sun_dir.x; u.sun_dir.y = sun_dir.y; u.sun_dir.z = sun_dir.z;
    u.sun_intensity.x = sun_intensity.x; u.sun_intensity.y = sun_intensity.y; u.sun_intensity.z = sun_intensity.z;
    u.num_clusters.x = NUM_CLUSTERS_X;
    u.num_clusters.y = NUM_CLUSTERS_Y;
    u.cluster_size_in_pixels.x = (float)width / (float)NUM_CLUSTERS_X;
    u.cluster_size_in_pixels.y = (float)height / (float)NUM_CLUSTERS_Y;
    return u;
}

inline tr_push_constants make_push_constants(const Mat4& proj_view, Vec3 view_position, uint32_t width, uint32_t height,
                                             uint64_t acceleration_structure_address = 0) {
    tr_push_constants pc;
    std::memset(&pc, 0, sizeof pc);
    pc.proj_view = proj_view.to_abi();
    pc.view_position.x = view_position.x; pc.view_position.y = view_position.y; pc.view_position.z = view_position.z;
    pc.framebuffer_size.x = width;
    pc.framebuffer_size.y = height;
    pc.acceleration_structure_address = acceleration_structure_address;
    return pc;
}

// src/main.rs:1728-1746: the side planes of the frustum from rows 3 + 0 and 3 + 1 of the perspective matrix
inline tr_culling_push_constants make_culling_push_constants(const Mat4& view, const Mat4& perspective) {
    const Vec3 fx = normalize({perspective.m[3][0] + perspective.m[0][0], perspective.m[3][1] + perspective.m[0][1], perspective.m[3][2] + perspective.m[0][2]});
    const Vec3 fy = normalize({perspective.m[3][0] + perspective.m[1][0], perspective.m[3][1] + perspective.m[1][1], perspective.m[3][2] + perspective.m[1][2]});
    tr_culling_push_constants c;
    std::memset(&c, 0, sizeof c);
    c.view = view.to_abi();
    c.frustum_x_xz.x = fx.x; c.frustum_x_xz.y = fx.z;
    c.frustum_y_yz.x = fy.y; c.frustum_y_yz.y = fy.z;
    c.z_near = Z_NEAR;
    return c;
}

// glam Mat4::inverse of the perspective matrix (src/main.rs:1502-1505), in double by Gauss-Jordan, rounded once
inline Mat4 inverse(const Mat4& a) {
    double w[4][8];
    for (int i = 0; i < 4; i++)
        for (int j = 0; j < 4; j++) {
            w[i][j] = a.m[i][j];
            w[i][4 + j] = i == j ? 1.0 : 0.0;
        }
    for (int col = 0; col < 4; col++) {
        int piv = col;
        for (int r = col + 1; r < 4; r++)
            if (std::fabs(w[r][col]) > std::fabs(w[piv][col])) piv = r;
        if (w[piv][col] == 0.0) throw std::domain_error("tr::inverse: singular matrix");
        for (int j = 0; j < 8; j++) std::swap(w[col][j], w[piv][j]);
        const double d = w[col][col];
        for (int j = 0; j < 8; j++) w[col][j] /= d;
        for (int r = 0; r < 4; r++) {
            if (r == col) continue;
            const double f = w[r][col];
            for (int j = 0; j < 8; j++) w[r][j] -= f * w[col][j];
        }
    }
    Mat4 o;
    for (int i = 0; i < 4; i++)
        for (int j = 0; j < 4; j++) o.m[i][j] = (float)w[i][4 + j];
    return o;
}

inline tr_write_cluster_data_push_constants make_write_cluster_data_push_constants(const Mat4& perspective, uint32_t width, uint32_t height) {
    tr_write_cluster_data_push_constants w;
    std::memset(&w, 0, sizeof w);
    w.inverse_perspective = inverse(perspective).to_abi();
    w.screen_dimensions.x = width;
    w.screen_dimensions.y = height;
    return w;
}

// src/main.rs:1785-1788: view_rotation = camera rotation inverse
inline tr_assign_lights_push_constants make_assign_lights_push_constants(const Mat4& view, Quat camera_rotation) {
    tr_assign_lights_push_constants a;
    std::memset(&a, 0, sizeof a);
    a.view_matrix = view.to_abi();
    const Quat q = inverse(camera_rotation);
    a.view_rotation.x = q.x; a.view_rotation.y = q.y; a.view_rotation.z = q.z; a.view_rotation.w = q.w;
    return a;
}

// Light::new_point, shared-structs/src/lib.rs:94-103
inline tr_light light_new_point(Vec3 position, Vec3 colour, float intensity) {
    tr_light l;
    std::memset(&l, 0, sizeof l);
    l.position_and_spotlight_epsilon.x = position.x; l.position_and_spotlight_epsilon.y = position.y; l.position_and_spotlight_epsilon.z = position.z;
    l.colour_emission_and_falloff_distance_sq.x = colour.x * intensity;
    l.colour_emission_and_falloff_distance_sq.y = colour.y * intensity;
    l.colour_emission_and_falloff_distance_sq.z = colour.z * intensity;
    l.colour_emission_and_falloff_distance_sq.w = intensity / 0.05f;   // distance_sq_at_strength(intensity, 0.05)
    return l;
}

// Light::new_spot, shared-structs/src/lib.rs:105-123
inline tr_light light_new_spot(Vec3 position, Vec3 colour, float intensity, Vec3 direction, float inner_angle_rad, float outer_angle_rad) {
    tr_light l = light_new_point(position, colour, intensity);
    l.position_and_spotlight_epsilon.w = std::cos(inner_angle_rad) - std::cos(outer_angle_rad);
    l.spotlight_direction_and_outer_angle.x = direction.x; l.spotlight_direction_and_outer_angle.y = direction.y; l.spotlight_direction_and_outer_angle.z = direction.z;
    l.spotlight_direction_and_outer_angle.w = outer_angle_rad;
    return l;
}

// BakedLottesTonemapperParams::from(LottesTonemapperParams::default()) (src/main.rs:506-510; colstodian is not part of
// the reference tree): the published Lottes parameterisation with contrast 1.6, shoulder 0.977, hdr_max 8, mid_in 0.18,
// mid_out 0.267 — the same numbers transmission_renderer_b200/host.py derives
inline tr_baked_lottes_tonemapper_params default_tonemap_params() {
    const double contrast = 1.6, shoulder = 0.977, hdr_max = 8.0, mid_in = 0.18, mid_out = 0.267;
    const double a = contrast, d = shoulder, ha = std::pow(hdr_max, a), ma = std::pow(mid_in, a), had = std::pow(ha, d), mad = std::pow(ma, d);
    tr_baked_lottes_tonemapper_params p;
    p.a = (float)a;
    p.b = (float)((-ma + ha * mid_out) / ((had - mad) * mid_out));
    p.c = (float)((had * ma - ha * mad * mid_out) / ((had - mad) * mid_out));
    p.d = (float)d;
    p.crosstalk = 4.0f;
    p.saturation = (float)contrast;
    p.cross_saturation = 16.0f;
    return p;
}

inline uint32_t mip_levels_for_size(uint32_t width, uint32_t height) {   // src/main.rs:2590-2592
    return (uint32_t)std::log2((float)(width < height ? width : height)) + 1u;
}
inline uint32_t dispatch_count(uint32_t num, uint32_t group_size) {      // src/main.rs:2639-2641
    return num == 0 ? 0 : (num - 1) / group_size + 1;
}
// image-band partition of SURVEY.md 8e: rows [floor(r H / N), floor((r + 1) H / N))
inline std::pair<uint32_t, uint32_t> band_rows(uint32_t height, uint32_t rank, uint32_t world_size) {
    return {(uint32_t)(((uint64_t)rank * height) / world_size), (uint32_t)(((uint64_t)(rank + 1) * height) / world_size)};
}

// Everything record() needs per frame, from one camera (src/main.rs:1186-1232, 1728-1746, 1785-1788)
inline tr_frame_params make_frame_params(const Camera& cam, uint32_t width, uint32_t height, const tr_baked_lottes_tonemapper_params& tonemap,
                                         uint32_t flags = 0, uint64_t acceleration_structure_address = 0) {
    const Mat4 perspective = perspective_matrix_reversed(width, height);
    tr_frame_params f;
    std::memset(&f, 0, sizeof f);
    f.culling = make_culling_push_constants(cam.view, perspective);
    f.assign_lights = make_assign_lights_push_constants(cam.view, cam.rotation);
    f.push_constants = make_push_constants(mul(perspective, cam.view), cam.position, width, height, acceleration_structure_address);
    f.tonemap = tonemap;
    f.flags = flags;
    return f;
}

// ---- errors: the reference propagates anyhow::Error with `?`; here a status other than TR_OK becomes an exception ----------
class Error : public std::runtime_error {
public:
    Error(int32_t status, const std::string& what) : std::runtime_error(what), status_(status) {}
    int32_t status() const { return status_; }

private:
    int32_t status_;
};
inline void check(int32_t status, const char* call) {
    if (status != TR_OK) throw Error(status, std::string(call) + ": " + tr_last_error());
}
#define TR_HOST_CHECK(call) ::tr::check((call), #call)

// ---- Renderer: owns a tr_ctx (Pipelines::new + DescriptorSets::allocate on construction, the LoopDestroyed clean-up on
// destruction, src/main.rs:1416-1445).  One per GPU / host thread.
class Renderer {
public:
    Renderer(uint32_t width, uint32_t height, int32_t device = 0, uint32_t flags = 0) : width_(width), height_(height) {
        tr_config cfg = {width, height, device, 0, 0, flags};
        TR_HOST_CHECK(tr_create(&cfg, &ctx_));
    }
    ~Renderer() {
        if (ctx_) tr_destroy(ctx_);
    }
    Renderer(const Renderer&) = delete;
    Renderer& operator=(const Renderer&) = delete;
    Renderer(Renderer&& o) noexcept : ctx_(o.ctx_), width_(o.width_), height_(o.height_) { o.ctx_ = nullptr; }

    tr_ctx* ctx() const { return ctx_; }
    uint32_t width() const { return width_; }
    uint32_t height() const { return height_; }

    // ModelStagingBuffers::upload (src/main.rs:2495-2560) and the descriptor writes of :715-828
    void set_mesh(const std::vector<float>& positions, const std::vector<float>& normals, const std::vector<float>& uvs,
                  const std::vector<uint32_t>& indices) {
        if (positions.size() % 3 || normals.size() != positions.size() || uvs.size() * 3 != positions.size() * 2)
            throw Error(TR_ERR_INVALID_ARG, "Renderer::set_mesh: positions / normals / uvs disagree about the vertex count");
        TR_HOST_CHECK(tr_set_mesh(ctx_, positions.data(), normals.data(), uvs.data(), (uint32_t)(positions.size() / 3), indices.data(), (uint32_t)indices.size()));
    }
    // vertex animation: positions and normals of vertices [first_vertex, first_vertex + n) in stream order; with ray queries,
    // update the top level (update_top_level_acceleration_structure_async) before the next frame
    void update_mesh_vertices(const std::vector<float>& positions, const std::vector<float>& normals, uint32_t first_vertex = 0) {
        if (positions.size() % 3 || normals.size() != positions.size())
            throw Error(TR_ERR_INVALID_ARG, "Renderer::update_mesh_vertices: positions / normals disagree about the vertex count");
        TR_HOST_CHECK(tr_update_mesh_vertices(ctx_, first_vertex, (uint32_t)(positions.size() / 3), positions.data(), normals.data()));
    }
    void set_instances(const std::vector<tr_instance>& v) { TR_HOST_CHECK(tr_set_instances(ctx_, v.data(), (uint32_t)v.size())); }
    // the instance write of --rotate-model (src/main.rs:1263-1345) with unchanged ids: new transforms for instances
    // [first, first + n) in stream order; with ray queries, update the top level (update_top_level_acceleration_structure_async)
    // before the next frame.  `transforms` may also point to device memory (tr_abi.h, "Device sources").
    void update_instance_transforms(const tr_packed_similarity* transforms, uint32_t n, uint32_t first = 0) {
        TR_HOST_CHECK(tr_update_instance_transforms(ctx_, first, n, transforms));
    }
    void update_instance_transforms(const std::vector<tr_packed_similarity>& v, uint32_t first = 0) {
        update_instance_transforms(v.empty() ? nullptr : v.data(), (uint32_t)v.size(), first);
    }
    void set_primitives(const std::vector<tr_primitive_info>& v) { TR_HOST_CHECK(tr_set_primitives(ctx_, v.data(), (uint32_t)v.size())); }
    void set_materials(const std::vector<tr_material_info>& v) { TR_HOST_CHECK(tr_set_materials(ctx_, v.data(), (uint32_t)v.size())); }
    void set_lights(const std::vector<tr_light>& v) { TR_HOST_CHECK(tr_set_lights(ctx_, v.empty() ? nullptr : v.data(), (uint32_t)v.size())); }
    void set_uniforms(const tr_uniforms& u) { TR_HOST_CHECK(tr_set_uniforms(ctx_, &u)); }
    // load_texture_from_gltf + ImageManager::push_image, src/model_loading.rs:340-379: level 0 of image `index` (RGBA8,
    // tightly packed), the mip chain built on the device in stream order (n_levels = 0: the full chain).  `rgba8` is read
    // during the call unless it is page-locked; then it must stay alive and unchanged until the stream has passed the call.
    void set_texture_async(uint32_t index, const std::vector<uint8_t>& rgba8, uint32_t w, uint32_t h, bool srgb, uint32_t n_levels = 0) {
        if (rgba8.size() != (size_t)w * h * 4) throw Error(TR_ERR_INVALID_ARG, "Renderer::set_texture_async: size");
        TR_HOST_CHECK(tr_set_texture_async(ctx_, index, rgba8.data(), w, h, srgb ? 1 : 0, n_levels));
    }
    void set_ggx_lut(const std::vector<uint8_t>& rgba8, uint32_t w, uint32_t h) {
        if (rgba8.size() != (size_t)w * h * 4) throw Error(TR_ERR_INVALID_ARG, "Renderer::set_ggx_lut: size");
        TR_HOST_CHECK(tr_set_ggx_lut(ctx_, rgba8.data(), w, h));
    }
    // src/main.rs:996-1166: new extent -> new targets, cluster sizes and cluster AABBs
    void resize(uint32_t width, uint32_t height) {
        TR_HOST_CHECK(tr_resize(ctx_, width, height));
        width_ = width;
        height_ = height;
    }
    void build_clusters() {   // src/main.rs:1498-1515
        const tr_write_cluster_data_push_constants pc = make_write_cluster_data_push_constants(perspective_matrix_reversed(width_, height_), width_, height_);
        TR_HOST_CHECK(tr_build_clusters(ctx_, &pc));
    }
    uint64_t build_acceleration_structures() {   // src/main.rs:577-658
        uint64_t address = 0;
        TR_HOST_CHECK(tr_build_acceleration_structures(ctx_, &address));
        return address;
    }
    // the same, built on the device in stream order without waiting for the GPU (also the rebuild after refits)
    uint64_t build_acceleration_structures_async() {
        uint64_t address = 0;
        TR_HOST_CHECK(tr_build_acceleration_structures_async(ctx_, &address));
        return address;
    }
    // update_top_level_acceleration_structure_from_instances, src/acceleration_structures.rs:188-263: after set_instances
    uint64_t update_top_level_acceleration_structure() {
        uint64_t address = 0;
        TR_HOST_CHECK(tr_update_top_level_acceleration_structure(ctx_, &address));
        return address;
    }
    // the same, built on the device in stream order without waiting for the GPU (the per-frame form, src/main.rs:1263-1345)
    uint64_t update_top_level_acceleration_structure_async() {
        uint64_t address = 0;
        TR_HOST_CHECK(tr_update_top_level_acceleration_structure_async(ctx_, &address));
        return address;
    }
    // record(), src/main.rs:1551-2263
    void frame(const tr_frame_params& f) { TR_HOST_CHECK(tr_frame(ctx_, &f)); }
    void sync() { TR_HOST_CHECK(tr_sync(ctx_)); }
    std::vector<uint8_t> read_srgb8() {
        std::vector<uint8_t> out((size_t)width_ * height_ * 4);
        TR_HOST_CHECK(tr_read_srgb8(ctx_, out.data()));
        return out;
    }
    std::vector<uint16_t> read_hdr() {
        std::vector<uint16_t> out((size_t)width_ * height_ * 4);
        TR_HOST_CHECK(tr_read_hdr(ctx_, out.data()));
        return out;
    }
    std::vector<uint32_t> read_visible_instances(uint32_t capacity) {
        std::vector<uint32_t> ids(capacity);
        uint32_t n = 0;
        TR_HOST_CHECK(tr_read_visible_instances(ctx_, ids.data(), capacity, &n));
        ids.resize(n);
        return ids;
    }
    // band sharding, SURVEY.md 8e
    void set_band(uint32_t y0, uint32_t y1) { TR_HOST_CHECK(tr_set_band(ctx_, y0, y1)); }
    void comm_init(const uint8_t id[TR_NCCL_UNIQUE_ID_BYTES], int32_t rank, int32_t n_ranks) { TR_HOST_CHECK(tr_comm_init(ctx_, id, rank, n_ranks)); }

private:
    friend class RendererGroup;   // tr_group_resize resizes the members
    tr_ctx* ctx_ = nullptr;
    uint32_t width_, height_;
};

// ---- RendererGroup: one Renderer per entry of `devices` (repeats allowed), joined into the bands of one frame
// (tr_group_*).  The reference's host is one thread with one queue (src/main.rs:243); this is how that thread drives up to 8
// GPUs.  Uploads and reads go to member(k) as to any Renderer; the frame goes through the group.
class RendererGroup {
public:
    RendererGroup(const std::vector<int32_t>& devices, uint32_t width, uint32_t height, uint32_t flags = 0) : width_(width), height_(height) {
        if (devices.empty() || devices.size() > 8) throw Error(TR_ERR_INVALID_ARG, "RendererGroup: 1 to 8 devices");
        members_.reserve(devices.size());
        for (int32_t d : devices) members_.emplace_back(width, height, d, flags);
        std::vector<tr_ctx*> ctxs;
        for (const Renderer& r : members_) ctxs.push_back(r.ctx());
        TR_HOST_CHECK(tr_group_create(ctxs.data(), (uint32_t)ctxs.size(), &group_));
    }
    ~RendererGroup() {   // the group first: a member is not destroyed while it belongs to one
        if (group_) tr_group_destroy(group_);
    }
    RendererGroup(const RendererGroup&) = delete;
    RendererGroup& operator=(const RendererGroup&) = delete;

    size_t size() const { return members_.size(); }
    Renderer& member(size_t k) { return members_.at(k); }
    tr_group* group() const { return group_; }

    void set_bands(const std::vector<uint32_t>& bounds) { TR_HOST_CHECK(tr_group_set_bands(group_, bounds.data(), (uint32_t)bounds.size())); }
    void resize(uint32_t width, uint32_t height) {   // src/main.rs:996-1166 on every member; equal-row bands again
        TR_HOST_CHECK(tr_group_resize(group_, width, height));
        width_ = width;
        height_ = height;
        for (Renderer& r : members_) {
            r.width_ = width;
            r.height_ = height;
        }
    }
    // record(), src/main.rs:1551-2263, across the members: one camera for all, or one tr_frame_params per member (each with
    // its own acceleration_structure_address when ray queries are on)
    void frame(const tr_frame_params& f) { frame(std::vector<tr_frame_params>(members_.size(), f)); }
    void frame(const std::vector<tr_frame_params>& per_member) {
        if (per_member.size() != members_.size()) throw Error(TR_ERR_INVALID_ARG, "RendererGroup::frame: one tr_frame_params per member");
        TR_HOST_CHECK(tr_group_frame(group_, per_member.data()));
    }
    void sync() { TR_HOST_CHECK(tr_group_sync(group_)); }
    // load member(source) only, then copy its scene into every other member, GPU to GPU in stream order
    // (tr_group_replicate_scene); returns every member's acceleration-structure handle (0: the source has no valid top level)
    std::vector<uint64_t> replicate_scene(uint32_t source = 0) {
        std::vector<uint64_t> addresses(members_.size());
        TR_HOST_CHECK(tr_group_replicate_scene(group_, source, addresses.data()));
        return addresses;
    }
    std::vector<uint8_t> read_srgb8() {   // the whole frame, every member's band
        std::vector<uint8_t> out((size_t)width_ * height_ * 4);
        TR_HOST_CHECK(tr_group_read_srgb8(group_, out.data()));
        return out;
    }

private:
    std::vector<Renderer> members_;
    tr_group* group_ = nullptr;
    uint32_t width_, height_;
};

}  // namespace tr
#endif
