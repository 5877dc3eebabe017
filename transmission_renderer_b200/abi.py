"""numpy mirrors of the `#[repr(C)]` structs in include/tr_abi.h.

Reference layouts: /root/reference/shared-structs/src/lib.rs (offsets as in
SURVEY.md Appendix A, verified there against the shipped SPIR-V).  Matrices are
stored column-major like glam::Mat4: ``arr['proj_view'][col][row]``; assign a
math-convention (row, col) numpy matrix ``M`` with ``= M.T``.
"""
import numpy as np


def _dt(fields, itemsize):
    names, formats, offsets = zip(*fields)
    return np.dtype({"names": list(names), "formats": list(formats), "offsets": list(offsets), "itemsize": itemsize})


MAT4 = ("<f4", (4, 4))
VEC4 = ("<f4", (4,))
VEC3 = ("<f4", (3,))
VEC2 = ("<f4", (2,))
UVEC2 = ("<u4", (2,))

push_constants = _dt(
    [("proj_view", MAT4, 0), ("view_position", VEC4, 64), ("framebuffer_size", UVEC2, 80),
     ("acceleration_structure_address", "<u8", 88)], 96)

uniforms = _dt(
    [("z_near", "<f4", 0), ("z_far", "<f4", 4), ("scale", "<f4", 8), ("bias", "<f4", 12),
     ("num_depth_slices", "<u4", 16), ("sun_dir", VEC4, 32), ("sun_intensity", VEC4, 48),
     ("cluster_size_in_pixels", VEC2, 64), ("num_clusters", UVEC2, 72), ("debug_clusters", "<u4", 80),
     ("ggx_lut_texture_index", "<u4", 84)], 96)

light = _dt(
    [("position_and_spotlight_epsilon", VEC4, 0), ("colour_emission_and_falloff_distance_sq", VEC4, 16),
     ("spotlight_direction_and_outer_angle", VEC4, 32)], 48)

material_info = _dt(
    [("textures", ("<i4", (9,)), 0), ("metallic_factor", "<f4", 36), ("roughness_factor", "<f4", 40),
     ("alpha_clipping_cutoff", "<f4", 44), ("diffuse_factor", VEC4, 48), ("emissive_factor", VEC4, 64),
     ("normal_map_scale", "<f4", 80), ("occlusion_strength", "<f4", 84), ("index_of_refraction", "<f4", 88),
     ("transmission_factor", "<f4", 92), ("thickness_factor", "<f4", 96), ("attenuation_distance", "<f4", 100),
     ("attenuation_colour", VEC4, 112), ("specular_factor", "<f4", 128), ("specular_colour_factor", VEC4, 144)], 160)

instance = _dt(
    [("translation_and_scale", VEC4, 0), ("rotation", VEC4, 16), ("primitive_id", "<u4", 32),
     ("material_id", "<u4", 36)], 48)

primitive_info = _dt(
    [("packed_bounding_sphere", VEC4, 0), ("draw_buffer_index", "<u4", 16), ("index_count", "<u4", 20),
     ("first_index", "<u4", 24), ("first_instance", "<u4", 28)], 32)

culling_push_constants = _dt(
    [("view", MAT4, 0), ("frustum_x_xz", VEC2, 64), ("frustum_y_yz", VEC2, 72), ("z_near", "<f4", 80)], 96)

cluster_aabb = _dt([("min", VEC4, 0), ("max", VEC4, 16)], 32)

write_cluster_data_push_constants = _dt([("inverse_perspective", MAT4, 0), ("screen_dimensions", UVEC2, 64)], 80)

assign_lights_push_constants = _dt([("view_matrix", MAT4, 0), ("view_rotation", VEC4, 64)], 80)

draw_indexed_indirect_command = _dt(
    [("index_count", "<u4", 0), ("instance_count", "<u4", 4), ("first_index", "<u4", 8), ("vertex_offset", "<i4", 12),
     ("first_instance", "<u4", 16)], 20)

baked_lottes_tonemapper_params = _dt(
    [("a", "<f4", 0), ("b", "<f4", 4), ("c", "<f4", 8), ("d", "<f4", 12), ("crosstalk", "<f4", 16),
     ("saturation", "<f4", 20), ("cross_saturation", "<f4", 24)], 28)

# glam-pbr contract batch forms
material_params = _dt(
    [("diffuse_colour", VEC3, 0), ("metallic", "<f4", 12), ("perceptual_roughness", "<f4", 16),
     ("index_of_refraction", "<f4", 20), ("specular_colour", VEC3, 24), ("specular_factor", "<f4", 36)], 40)

basic_brdf_params = _dt(
    [("normal", VEC3, 0), ("light", VEC3, 12), ("light_intensity", VEC3, 24), ("view", VEC3, 36),
     ("material_params", material_params, 48)], 88)

brdf_result = _dt([("diffuse", VEC3, 0), ("specular", VEC3, 12)], 24)

transmission_btdf_params = _dt(
    [("material_params", material_params, 0), ("normal", VEC3, 40), ("view", VEC3, 52), ("light", VEC3, 64)], 76)

point_light_params = _dt(
    [("normal", VEC3, 0), ("view", VEC3, 12), ("position", VEC3, 24), ("light_position", VEC3, 36),
     ("light_colour", VEC3, 48), ("material_params", material_params, 60)], 100)

point_light_result = _dt([("diffuse", VEC3, 0), ("specular", VEC3, 12), ("transmission", VEC3, 24)], 36)

ibl_volume_refraction_params = _dt(
    [("material_params", material_params, 0), ("framebuffer_size_x", "<u4", 40), ("normal", VEC3, 44),
     ("view", VEC3, 56), ("position", VEC3, 68), ("thickness", "<f4", 80), ("model_scale", "<f4", 84),
     ("attenuation_distance", "<f4", 88), ("attenuation_colour", VEC3, 92)], 104)

frame_params = _dt(
    [("culling", culling_push_constants, 0), ("assign_lights", assign_lights_push_constants, 96),
     ("push_constants", push_constants, 176), ("tonemap", baked_lottes_tonemapper_params, 272),
     ("flags", "<u4", 300)], 304)

frame_times = _dt(
    [(n, "<f4", 4 * i) for i, n in enumerate(
        ["cull_ms", "assign_lights_ms", "visibility_ms", "shade_opaque_ms", "allgather_ms", "mips_ms",
         "shade_transmission_ms", "tonemap_ms", "total_ms"])], 36)

TR_MAX_LIGHTS_PER_CLUSTER = 128
TR_FLAG_HDR_F32_DEBUG = 1
TR_FRAME_SKIP_TONEMAP = 1
TR_FRAME_SKIP_VISIBILITY = 2
TR_LAYER_OPAQUE = 0
TR_LAYER_TRANSMISSIVE = 1

STATUS_NAMES = {0: "TR_OK", -1: "TR_ERR_INVALID_ARG", -2: "TR_ERR_UNSUPPORTED", -3: "TR_ERR_CUDA",
                -4: "TR_ERR_NCCL", -5: "TR_ERR_OOM", -6: "TR_ERR_STATE"}


def default_material(n=1):
    """MaterialInfo defaults of the reference's loader (src/model_loading.rs:293-332)."""
    m = np.zeros(n, dtype=material_info)
    m["textures"] = -1
    m["metallic_factor"] = 1.0
    m["roughness_factor"] = 1.0
    m["alpha_clipping_cutoff"] = 0.5
    m["diffuse_factor"] = 1.0
    m["normal_map_scale"] = 1.0
    m["occlusion_strength"] = 1.0
    m["index_of_refraction"] = 1.5
    m["transmission_factor"] = 0.0
    m["thickness_factor"] = 0.0
    m["attenuation_distance"] = np.inf
    m["attenuation_colour"] = (1.0, 1.0, 1.0, 0.0)
    m["specular_factor"] = 1.0
    m["specular_colour_factor"] = (1.0, 1.0, 1.0, 0.0)
    return m

# the top level as tr_read_top_level_acceleration_structure returns it (csrc/tr_device_accel.cuh AccelNode, AccelInstance);
# c0 / c1 >= 0: inner node, < 0: leaf ~(first | (count - 1) << 28)
accel_node = _dt([("lo0", VEC3, 0), ("hi0", VEC3, 12), ("lo1", VEC3, 24), ("hi1", VEC3, 36), ("c0", "<i4", 48), ("c1", "<i4", 52),
                  ("pad", ("<u4", (2,)), 56)], 64)
accel_instance = _dt([("translation", VEC3, 0), ("inv_scale", "<f4", 12), ("conj_rotation", VEC4, 16), ("lo", VEC3, 32),
                      ("hi", VEC3, 44), ("blas_root", "<u4", 56), ("tri_base", "<u4", 60)], 64)
