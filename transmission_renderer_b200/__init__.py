"""transmission_renderer_b200 — B200-native per-pixel light-transport path of
expenses/transmission-renderer behind a C ABI (include/tr_abi.h).

The product is `libtr.so` (hand-written sm_100a CUDA, built in-tree by
`csrc/build.py`).  This package is only the thin host-side mirror of that ABI:
numpy struct layouts (`abi`), the host inputs the reference computes on the CPU
(`host`), procedural scenes (`scenes`) and a `Renderer` wrapper whose methods map
1:1 onto the `tr_*` entry points.  There is NO CPU fallback: if the library or a
CUDA device is missing, every call raises.
"""
import ctypes as C
import os

from . import abi, host  # noqa: F401

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("TR_LIB") or os.path.join(_HERE, "libtr.so")  # TR_LIB: an experimental build (csrc/build.py --out=)
_LIB = None

# every symbol include/tr_abi.h declares (checked by tests/test_abi_symbols.py)
EXPORTS = [
    "tr_create", "tr_destroy", "tr_resize", "tr_set_band", "tr_last_error", "tr_version", "tr_set_stream", "tr_sync",
    "tr_set_instances", "tr_update_instance_transforms", "tr_set_primitives", "tr_set_materials", "tr_set_lights", "tr_set_uniforms", "tr_set_ggx_lut", "tr_set_texture", "tr_set_texture_async",
    "tr_read_texture_level",
    "tr_set_mesh", "tr_update_mesh_vertices", "tr_read_chunk_spheres", "tr_build_acceleration_structures", "tr_build_acceleration_structures_async",
    "tr_update_top_level_acceleration_structure", "tr_update_top_level_acceleration_structure_async", "tr_trace_shadow_rays",
    "tr_read_shadow_mask", "tr_read_top_level_acceleration_structure", "tr_read_bottom_level_acceleration_structures", "tr_cull", "tr_build_clusters", "tr_assign_lights", "tr_visibility", "tr_shade_opaque",
    "tr_allgather_opaque", "tr_generate_mips", "tr_shade_transmission", "tr_tonemap", "tr_frame", "tr_set_gbuffer",
    "tr_read_gbuffer", "tr_set_opaque_frame", "tr_set_hdr", "tr_set_cluster_lights", "tr_read_visible_instances",
    "tr_read_instance_counts", "tr_read_draws", "tr_read_cluster_aabbs", "tr_read_cluster_lights", "tr_read_hdr",
    "tr_read_hdr_f32", "tr_read_pyramid_level", "tr_read_srgb8", "tr_read_srgb8_async", "tr_wait_readback", "tr_mip_levels", "tr_enable_timing",
    "tr_begin_frame", "tr_read_frame_times", "tr_read_pass_totals", "tr_eval_basic_brdf", "tr_eval_transmission_btdf", "tr_eval_point_light", "tr_eval_ibl_volume_refraction",
    "tr_set_bands", "tr_comm_unique_id", "tr_comm_init", "tr_comm_destroy", "tr_peer_export", "tr_peer_attach", "tr_device_buffer",
    "tr_launch_count", "tr_raster_stats", "tr_measure_fp32_peak", "tr_measure_hbm_copy",
    "tr_group_create", "tr_group_destroy", "tr_group_set_bands", "tr_group_resize", "tr_group_frame", "tr_group_sync",
    "tr_group_read_srgb8", "tr_group_replicate_scene",
]


class TrError(RuntimeError):
    def __init__(self, status, message):
        super().__init__(f"{abi.STATUS_NAMES.get(status, status)}: {message}")
        self.status = status


def lib():
    """Loads libtr.so; raises loudly if it has not been built (python -m transmission_renderer_b200.csrc.build)."""
    global _LIB
    if _LIB is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(f"{LIB_PATH} is missing: the CUDA library is the product and has no substitute; "
                              "build it with `python -m transmission_renderer_b200.csrc.build`")
        _LIB = C.CDLL(LIB_PATH)
        _LIB.tr_last_error.restype = C.c_char_p
        _LIB.tr_version.restype = C.c_char_p
        for name in EXPORTS:
            fn = getattr(_LIB, name)
            if name not in ("tr_last_error", "tr_version"):
                fn.restype = C.c_int32
    return _LIB


def _check(status):
    if status != 0:
        raise TrError(status, lib().tr_last_error().decode())


from .renderer import Renderer, RendererGroup  # noqa: E402,F401
