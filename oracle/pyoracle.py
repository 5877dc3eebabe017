"""ctypes front-end of the CPU oracle (oracle/liboracle.so).

TEST INFRASTRUCTURE ONLY — importable from tests/, __graft_entry__.smoke() and
bench.py's cpu_baseline / --impl reference legs.  The product package never
imports this module.  Parity: pinned to the reference's compiled shader modules (see oracle/oracle.h).
"""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

from transmission_renderer_b200 import abi

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None
_VARIANT = "parity"   # "parity": -O2 -ffp-contract=off (the checker); "o3": -O3 -march=native, a timing variant only


def build(force=False, variant="parity"):
    if variant != "parity":
        return _build_o3(force)
    so = os.path.join(_HERE, "liboracle.so")
    srcs = [os.path.join(_HERE, f) for f in os.listdir(_HERE) if f.endswith((".c", ".h")) and not f.startswith("spv_")]
    srcs.append(os.path.join(_HERE, "..", "include", "tr_abi.h"))
    if force or not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
        subprocess.check_call(["make", "-C", _HERE, "-s", "liboracle.so"])
    return so


_O3_DIR = None


def _build_o3(force):
    """The -O3 -march=native timing variant is built when it is asked for, for the CPU it runs on, in a temporary
    directory of this process (the source tree may be read-only)."""
    global _O3_DIR
    if _O3_DIR is None:
        _O3_DIR = tempfile.TemporaryDirectory(prefix="tr_oracle_o3_")
    so = os.path.join(_O3_DIR.name, "liboracle_o3.so")
    if force or not os.path.exists(so):
        subprocess.check_call(["make", "-C", _HERE, "-s", so, "O3_SO=" + so])
    return so


def select_variant(variant):
    """Swap the library behind this module (bench.py times the -O3 -march=native build next to the parity build)."""
    global _LIB, _VARIANT
    if variant != _VARIANT:
        build(variant=variant)
        _VARIANT, _LIB = variant, None


class Pyramid(C.Structure):
    _fields_ = [("levels", C.c_uint32), ("width", C.c_uint32 * 16), ("height", C.c_uint32 * 16),
                ("data", C.c_void_p * 16)]


class Lut(C.Structure):
    _fields_ = [("width", C.c_uint32), ("height", C.c_uint32), ("rgba8", C.c_void_p)]


class GBuffer(C.Structure):
    _fields_ = [("width", C.c_uint32), ("height", C.c_uint32), ("depth", C.c_void_p), ("normal", C.c_void_p),
                ("uv", C.c_void_p), ("material_id", C.c_void_p), ("scale", C.c_void_p), ("position", C.c_void_p),
                ("duv", C.c_void_p), ("ddepth", C.c_void_p)]


class Texture(C.Structure):
    _fields_ = [("width", C.c_uint32), ("height", C.c_uint32), ("levels", C.c_uint32), ("srgb", C.c_uint32),
                ("data", C.c_void_p * 16)]


class Scene(C.Structure):
    _fields_ = [("pc", C.c_void_p), ("uniforms", C.c_void_p), ("materials", C.c_void_p), ("n_materials", C.c_uint32),
                ("lights", C.c_void_p), ("n_lights", C.c_uint32), ("cluster_light_counts", C.c_void_p),
                ("cluster_light_indices", C.c_void_p), ("n_clusters", C.c_uint32), ("textures", C.c_void_p),
                ("n_textures", C.c_uint32), ("accel", C.c_void_p)]


class Mesh(C.Structure):
    _fields_ = [("positions", C.c_void_p), ("normals", C.c_void_p), ("uvs", C.c_void_p), ("indices", C.c_void_p),
                ("n_vertices", C.c_uint32), ("n_indices", C.c_uint32)]


def lib():
    global _LIB
    if _LIB is None:
        _LIB = C.CDLL(build(variant=_VARIANT))
        _LIB.orc_log2_spec.restype = C.c_float
        _LIB.orc_log2_spec.argtypes = [C.c_float]
        _LIB.orc_linear_depth.restype = C.c_float
        _LIB.orc_linear_depth.argtypes = [C.c_void_p, C.c_float]
        _LIB.orc_get_depth_slice.restype = C.c_uint32
        _LIB.orc_get_depth_slice.argtypes = [C.c_void_p, C.c_float]
        _LIB.orc_slice_to_depth.restype = C.c_float
        _LIB.orc_slice_to_depth.argtypes = [C.c_void_p, C.c_uint32]
        _LIB.orc_mip_levels_for_size.restype = C.c_uint32
        _LIB.orc_srgb8_encode.restype = C.c_uint8
        _LIB.orc_srgb8_encode.argtypes = [C.c_float]
        _LIB.orc_num_threads.restype = C.c_int
        _LIB.orc_d_ggx.restype = C.c_float
        _LIB.orc_d_ggx.argtypes = [C.c_float, C.c_float]
        _LIB.orc_v_smith_ggx_correlated.restype = C.c_float
        _LIB.orc_v_smith_ggx_correlated.argtypes = [C.c_float, C.c_float, C.c_float]
        _LIB.orc_ior_to_dielectric_f0.restype = C.c_float
        _LIB.orc_ior_to_dielectric_f0.argtypes = [C.c_float]
    return _LIB


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _c(a, dtype):
    return np.ascontiguousarray(a, dtype=dtype)


def num_threads():
    return int(lib().orc_num_threads())


def set_num_threads(n):
    lib().orc_set_num_threads(C.c_int(n))


# ---- fp16 helpers (numpy's float16 conversion is IEEE RNE as well) -------
def f16_bits(a):
    return np.asarray(a, dtype=np.float32).astype(np.float16).view(np.uint16)


def f16_to_f32(bits):
    return np.asarray(bits, dtype=np.uint16).view(np.float16).astype(np.float32)


# ---- glam-pbr batch evaluators --------------------------------------------
def eval_basic_brdf(params):
    params = _c(params, abi.basic_brdf_params)
    out = np.zeros(params.shape[0], dtype=abi.brdf_result)
    lib().orc_eval_basic_brdf(C.c_uint32(params.shape[0]), _p(params), _p(out))
    return out


def eval_transmission_btdf(params):
    params = _c(params, abi.transmission_btdf_params)
    out = np.zeros((params.shape[0], 3), dtype=np.float32)
    lib().orc_eval_transmission_btdf(C.c_uint32(params.shape[0]), _p(params), _p(out))
    return out


def eval_point_light(params):
    params = _c(params, abi.point_light_params)
    out = np.zeros(params.shape[0], dtype=abi.point_light_result)
    lib().orc_eval_point_light(C.c_uint32(params.shape[0]), _p(params), _p(out))
    return out


def make_pyramid_struct(levels):
    """levels: list of (h, w, 4) uint16 arrays."""
    p = Pyramid()
    p.levels = len(levels)
    keep = []
    for i, l in enumerate(levels):
        l = _c(l, np.uint16)
        keep.append(l)
        p.height[i], p.width[i] = l.shape[0], l.shape[1]
        p.data[i] = l.ctypes.data
    return p, keep


def make_lut_struct(rgba8):
    rgba8 = _c(rgba8, np.uint8)
    l = Lut()
    l.height, l.width = rgba8.shape[0], rgba8.shape[1]
    l.rgba8 = rgba8.ctypes.data
    return l, rgba8


def eval_ibl_volume_refraction(proj_view, params, levels, lut_rgba8):
    params = _c(params, abi.ibl_volume_refraction_params)
    pv = _c(np.asarray(proj_view, dtype=np.float32).T, np.float32)  # column-major
    pyr, keep = make_pyramid_struct(levels)
    lut, keep2 = make_lut_struct(lut_rgba8)
    out = np.zeros((params.shape[0], 3), dtype=np.float32)
    lib().orc_eval_ibl_volume_refraction(C.c_uint32(params.shape[0]), _p(pv), _p(params), C.byref(pyr), C.byref(lut),
                                         _p(out))
    return out


def sample_pyramid(levels, u, v, lod):
    pyr, keep = make_pyramid_struct(levels)
    fn = lib().orc_sample_pyramid

    class V3(C.Structure):
        _fields_ = [("x", C.c_float), ("y", C.c_float), ("z", C.c_float)]

    fn.restype = V3
    fn.argtypes = [C.c_void_p, C.c_float, C.c_float, C.c_float]
    r = fn(C.addressof(pyr), u, v, lod)
    return np.array([r.x, r.y, r.z], dtype=np.float32)


def sample_lut(lut_rgba8, nov, roughness):
    lut, keep = make_lut_struct(lut_rgba8)
    fn = lib().orc_sample_lut

    class V2(C.Structure):
        _fields_ = [("x", C.c_float), ("y", C.c_float)]

    fn.restype = V2
    fn.argtypes = [C.c_void_p, C.c_float, C.c_float]
    r = fn(C.addressof(lut), nov, roughness)
    return np.array([r.x, r.y], dtype=np.float32)


# ---- mip chain ---------------------------------------------------------------
def mip_levels_for_size(w, h):
    return int(lib().orc_mip_levels_for_size(C.c_uint32(w), C.c_uint32(h)))


def build_pyramid(mip0_bits):
    """mip0_bits: (h, w, 4) uint16 RGBA16F.  Returns the list of all levels."""
    mip0_bits = _c(mip0_bits, np.uint16)
    h, w = mip0_bits.shape[:2]
    n = mip_levels_for_size(w, h)
    levels = [mip0_bits]
    for _ in range(1, n):
        src = levels[-1]
        sh, sw = src.shape[:2]
        dh, dw = max(1, sh // 2), max(1, sw // 2)
        dst = np.zeros((dh, dw, 4), dtype=np.uint16)
        lib().orc_downsample_level(_p(src), C.c_uint32(sw), C.c_uint32(sh), _p(dst), C.c_uint32(dw), C.c_uint32(dh))
        levels.append(dst)
    return levels


# ---- compute entry points -------------------------------------------------------
def frustum_culling(instances, primitives, culling_pc):
    instances = _c(instances, abi.instance)
    primitives = _c(primitives, abi.primitive_info)
    culling_pc = _c(culling_pc, abi.culling_push_constants)
    counts = np.zeros(len(primitives), dtype=np.uint32)
    visible = np.zeros(max(1, len(instances)), dtype=np.uint32)
    n_visible = C.c_uint32(0)
    lib().orc_frustum_culling(_p(instances), C.c_uint32(len(instances)), _p(primitives), C.c_uint32(len(primitives)),
                              _p(culling_pc), _p(counts), _p(visible), C.byref(n_visible))
    return counts, visible[: n_visible.value].copy()


def demultiplex_draws(primitives, instance_counts):
    primitives = _c(primitives, abi.primitive_info)
    instance_counts = _c(instance_counts, np.uint32)
    n = len(primitives)
    draws = [np.zeros(max(1, n), dtype=abi.draw_indexed_indirect_command) for _ in range(4)]
    ptrs = (C.c_void_p * 4)(*[d.ctypes.data for d in draws])
    counts = np.zeros(4, dtype=np.uint32)
    lib().orc_demultiplex_draws(_p(primitives), _p(instance_counts), C.c_uint32(n), ptrs, _p(counts))
    return [d[: counts[i]].copy() for i, d in enumerate(draws)], counts


def write_cluster_data(uniforms, wc_pc, nz=16):
    uniforms = _c(uniforms, abi.uniforms)
    wc_pc = _c(wc_pc, abi.write_cluster_data_push_constants)
    nx, ny = int(uniforms["num_clusters"][0, 0]), int(uniforms["num_clusters"][0, 1])
    out = np.zeros(nx * ny * nz, dtype=abi.cluster_aabb)
    lib().orc_write_cluster_data(_p(uniforms), _p(wc_pc), C.c_uint32(nz), _p(out))
    return out


def assign_lights_to_clusters(lights, clusters, al_pc):
    lights = _c(lights, abi.light)
    clusters = _c(clusters, abi.cluster_aabb)
    al_pc = _c(al_pc, abi.assign_lights_push_constants)
    n = len(clusters)
    counts = np.zeros(n, dtype=np.uint32)
    indices = np.zeros(n * abi.TR_MAX_LIGHTS_PER_CLUSTER, dtype=np.uint32)
    lib().orc_assign_lights_to_clusters(_p(lights), C.c_uint32(len(lights)), _p(clusters), C.c_uint32(n), _p(al_pc),
                                        _p(counts), _p(indices))
    return counts, indices


def mat4_inverse(m_colmajor):
    m = _c(m_colmajor, np.float32).reshape(4, 4)
    out = np.zeros((4, 4), dtype=np.float32)
    lib().orc_mat4_inverse(_p(m), _p(out))
    return out


# ---- fragment stage ---------------------------------------------------------------
class _Keep:
    pass


def _gbuffer_struct(g, w, h):
    k = _Keep()
    k.depth = _c(g["depth"], np.float32)
    k.normal = _c(g["normal"], np.float32)
    k.uv = _c(g["uv"], np.float32) if g.get("uv") is not None else None
    k.mat = _c(g["material_id"], np.uint32)
    k.scale = _c(g["scale"], np.float32) if g.get("scale") is not None else None
    k.pos = _c(g["position"], np.float32) if g.get("position") is not None else None
    k.duv = _c(g["duv"], np.float32) if g.get("duv") is not None else None
    k.ddepth = _c(g["ddepth"], np.float32) if g.get("ddepth") is not None else None
    s = GBuffer(w, h, k.depth.ctypes.data, k.normal.ctypes.data, k.uv.ctypes.data if k.uv is not None else None,
                k.mat.ctypes.data, k.scale.ctypes.data if k.scale is not None else None,
                k.pos.ctypes.data if k.pos is not None else None, k.duv.ctypes.data if k.duv is not None else None,
                k.ddepth.ctypes.data if k.ddepth is not None else None)
    return s, k


def make_texture_array(textures):
    """textures: list of dict(levels=[(h, w, 4) uint8 ...], srgb=bool).  Returns (ctypes array, keep-alive)."""
    arr = (Texture * max(len(textures), 1))()
    keep = []
    for i, t in enumerate(textures):
        lv = [_c(l, np.uint8) for l in t["levels"]]
        keep.append(lv)
        arr[i].height, arr[i].width = lv[0].shape[0], lv[0].shape[1]
        arr[i].levels = len(lv)
        arr[i].srgb = 1 if t["srgb"] else 0
        for k, l in enumerate(lv):
            arr[i].data[k] = l.ctypes.data
    return arr, keep


def sample_texture(texture, uv, duv_dx, duv_dy):
    """uv, duv_dx, duv_dy: (n, 2).  Returns (n, 4) float32."""
    arr, keep = make_texture_array([texture])
    uv, dx, dy = (_c(a, np.float32).reshape(-1, 2) for a in (uv, duv_dx, duv_dy))
    L = lib()
    out = np.zeros((len(uv), 4), np.float32)

    class V2(C.Structure):
        _fields_ = [("x", C.c_float), ("y", C.c_float)]

    class V4(C.Structure):
        _fields_ = [("x", C.c_float), ("y", C.c_float), ("z", C.c_float), ("w", C.c_float)]
    L.orc_sample_texture.restype = V4
    L.orc_sample_texture.argtypes = [C.c_void_p, V2, V2, V2]
    for i in range(len(uv)):
        r = L.orc_sample_texture(C.addressof(arr[0]), V2(*uv[i]), V2(*dx[i]), V2(*dy[i]))
        out[i] = (r.x, r.y, r.z, r.w)
    return out


def _scene_struct(sc):
    k = _Keep()
    k.pc = _c(sc["push_constants"], abi.push_constants)
    k.u = _c(sc["uniforms"], abi.uniforms)
    k.m = _c(sc["materials"], abi.material_info)
    k.l = _c(sc["lights"], abi.light) if len(sc["lights"]) else np.zeros(1, dtype=abi.light)
    k.cc = _c(sc["cluster_light_counts"], np.uint32)
    k.ci = _c(sc["cluster_light_indices"], np.uint32)
    k.tex, k.tex_keep = make_texture_array(sc.get("textures") or [])
    n_tex = len(sc.get("textures") or [])
    s = Scene(k.pc.ctypes.data, k.u.ctypes.data, k.m.ctypes.data, len(k.m), k.l.ctypes.data, len(sc["lights"]),
              k.cc.ctypes.data, k.ci.ctypes.data, len(k.cc), C.addressof(k.tex) if n_tex else None, n_tex,
              sc["accel"].handle if sc.get("accel") is not None else None)
    return s, k


# ---- ray-queried shadows (oracle/shadow.c) ----------------------------------------
class Accel:
    """orc_accel: bottom-level trees per primitive + the top-level set of instances with draw_buffer_index < 2."""

    def __init__(self, mesh, instances, primitives):
        L = lib()
        L.orc_accel_build.restype = C.c_void_p
        L.orc_accel_instance_count.argtypes = [C.c_void_p]
        L.orc_accel_instance_count.restype = C.c_uint32
        self._keep = [_c(mesh["positions"], np.float32), _c(mesh["normals"], np.float32), _c(mesh["uvs"], np.float32),
                      _c(mesh["indices"], np.uint32), _c(instances, abi.instance), _c(primitives, abi.primitive_info)]
        pos, nrm, uv, idx, inst, prims = self._keep
        m = Mesh(pos.ctypes.data, nrm.ctypes.data, uv.ctypes.data, idx.ctypes.data, len(pos), len(idx))
        self.handle = L.orc_accel_build(C.byref(m), _p(inst), C.c_uint32(len(inst)), _p(prims), C.c_uint32(len(prims)))
        self.n_instances = L.orc_accel_instance_count(self.handle)

    def __del__(self):
        try:
            if self.handle:
                L = lib()
                L.orc_accel_free.argtypes = [C.c_void_p]
                L.orc_accel_free(self.handle)
                self.handle = None
        except Exception:
            pass

    def trace(self, origins, directions, t_max, brute=False):
        """(n,3), (n,3), (n,) -> (n,) uint8, 1 = lit, 0 = occluded (trace_shadow_ray, lighting.rs:97-125)."""
        o, d, t = _c(origins, np.float32).reshape(-1, 3), _c(directions, np.float32).reshape(-1, 3), _c(t_max, np.float32).reshape(-1)
        out = np.zeros(len(o), np.uint8)
        L = lib()
        L.orc_trace_shadow_rays.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
        L.orc_trace_shadow_rays(self.handle, len(o), o.ctypes.data, d.ctypes.data, t.ctypes.data, 1 if brute else 0, out.ctypes.data)
        return out


def slab_test(origin, direction, t_min, t_max, lo, hi):
    """The fp32 ray/box interval test of the shadow definition (oracle/shadow.c slab)."""
    a = [np.ascontiguousarray(x, np.float32) for x in (origin, direction, lo, hi)]
    L = lib()
    L.orc_slab_test.argtypes = [C.c_void_p, C.c_void_p, C.c_float, C.c_float, C.c_void_p, C.c_void_p]
    return bool(L.orc_slab_test(a[0].ctypes.data, a[1].ctypes.data, float(t_min), float(t_max), a[2].ctypes.data, a[3].ctypes.data))


def shadow_mask_frame(gbuffer, scene, y0=0, y1=None):
    """(5, h, w) uint32: occluded-ray bits per pixel (planes 0-3: position in the cluster's light list, plane 4: the sun)."""
    pc = scene["push_constants"]
    w, h = int(pc["framebuffer_size"][0, 0]), int(pc["framebuffer_size"][0, 1])
    y1 = h if y1 is None else y1
    g, kg = _gbuffer_struct(gbuffer, w, h)
    s, ks = _scene_struct(scene)
    out = np.zeros((5, h, w), np.uint32)
    lib().orc_shadow_mask_frame(C.byref(g), C.byref(s), C.c_uint32(y0), C.c_uint32(y1), _p(out))
    return out


def shade_opaque_frame(gbuffer, scene, y0=0, y1=None):
    """Returns (hdr_f32 (h,w,4), hdr_f16 bits (h,w,4)); the sampled opaque target equals hdr_f16."""
    pc = scene["push_constants"]
    w, h = int(pc["framebuffer_size"][0, 0]), int(pc["framebuffer_size"][0, 1])
    y1 = h if y1 is None else y1
    g, kg = _gbuffer_struct(gbuffer, w, h)
    s, ks = _scene_struct(scene)
    hdr32 = np.zeros((h, w, 4), dtype=np.float32)
    hdr16 = np.zeros((h, w, 4), dtype=np.uint16)
    lib().orc_shade_opaque_frame(C.byref(g), C.byref(s), C.c_uint32(y0), C.c_uint32(y1), _p(hdr32), _p(hdr16), None)
    return hdr32, hdr16


def shade_transmission_frame(gbuffer, scene, levels, lut_rgba8, hdr32, hdr16, y0=0, y1=None):
    """LOADs and updates hdr32 / hdr16 in place (copies are returned)."""
    pc = scene["push_constants"]
    w, h = int(pc["framebuffer_size"][0, 0]), int(pc["framebuffer_size"][0, 1])
    y1 = h if y1 is None else y1
    g, kg = _gbuffer_struct(gbuffer, w, h)
    s, ks = _scene_struct(scene)
    pyr, k1 = make_pyramid_struct(levels)
    lut, k2 = make_lut_struct(lut_rgba8)
    hdr32 = np.array(hdr32, dtype=np.float32, copy=True)
    hdr16 = np.array(hdr16, dtype=np.uint16, copy=True)
    lib().orc_shade_transmission_frame(C.byref(g), C.byref(s), C.byref(pyr), C.byref(lut), C.c_uint32(y0),
                                       C.c_uint32(y1), _p(hdr32), _p(hdr16))
    return hdr32, hdr16


def tonemap_frame(hdr16, params, y0=0, y1=None):
    hdr16 = _c(hdr16, np.uint16)
    h, w = hdr16.shape[:2]
    y1 = h if y1 is None else y1
    params = _c(params, abi.baked_lottes_tonemapper_params)
    out = np.zeros((h, w, 4), dtype=np.uint8)
    lib().orc_tonemap_frame(_p(hdr16), C.c_uint32(w), C.c_uint32(h), C.c_uint32(y0), C.c_uint32(y1), _p(params), _p(out))
    return out


def visibility(mesh, instances, primitives, visible_ids, push_constants, y0=0, y1=None, derivatives=False,
               materials=None, textures=None):
    """mesh: dict(positions (n,3), normals (n,3), uvs (n,2), indices (m,)).  Returns two G-buffer dicts; with
    derivatives=True each also carries the duv (h,w,4) / ddepth (h,w,2) forward-difference planes."""
    pos = _c(mesh["positions"], np.float32)
    nrm = _c(mesh["normals"], np.float32)
    uvs = _c(mesh["uvs"], np.float32)
    idx = _c(mesh["indices"], np.uint32)
    m = Mesh(pos.ctypes.data, nrm.ctypes.data, uvs.ctypes.data, idx.ctypes.data, len(pos), len(idx))
    instances = _c(instances, abi.instance)
    primitives = _c(primitives, abi.primitive_info)
    visible_ids = _c(visible_ids, np.uint32)
    pc = _c(push_constants, abi.push_constants)
    w, h = int(pc["framebuffer_size"][0, 0]), int(pc["framebuffer_size"][0, 1])
    y1 = h if y1 is None else y1
    layers = []
    for _ in range(2):
        layers.append(dict(depth=np.zeros((h, w), np.float32), normal=np.zeros((h, w, 3), np.float32),
                           uv=np.zeros((h, w, 2), np.float32), material_id=np.full((h, w), 0xFFFFFFFF, np.uint32),
                           scale=np.zeros((h, w), np.float32), position=None,
                           duv=np.zeros((h, w, 4), np.float32) if derivatives else None,
                           ddepth=np.zeros((h, w, 2), np.float32) if derivatives else None))
    a, b = layers
    mats = None if materials is None else _c(materials, abi.material_info)
    tex_arr, tex_keep = make_texture_array(textures or [])
    lib().orc_visibility(C.byref(m), _p(instances), C.c_uint32(len(instances)), _p(primitives),
                         C.c_uint32(len(primitives)), _p(visible_ids), C.c_uint32(len(visible_ids)), _p(pc),
                         C.c_uint32(y0), C.c_uint32(y1), _p(a["depth"]), _p(a["normal"]), _p(a["uv"]),
                         _p(a["material_id"]), _p(b["depth"]), _p(b["normal"]), _p(b["uv"]), _p(b["material_id"]),
                         _p(b["scale"]), _p(a["duv"]), _p(a["ddepth"]), _p(b["duv"]), _p(b["ddepth"]),
                         _p(mats), C.c_void_p(C.addressof(tex_arr)) if textures else None, C.c_uint32(len(textures or [])))
    a["scale"] = None
    return a, b


class ShadePathRunner:
    """The per-pixel shade path (fragment -> mip chain -> fragment_transmission -> tonemap) over rows
    [y0, y1) with every buffer preallocated, so a caller can time just the oracle's arithmetic.
    Used by bench.py's cpu_baseline / --impl reference legs (the CPU baseline is this port, all host
    threads via OpenMP)."""

    def __init__(self, g0, g1, scene, lut_rgba8, tonemap_params, opaque_full16=None):
        pc = scene["push_constants"]
        self.w, self.h = int(pc["framebuffer_size"][0, 0]), int(pc["framebuffer_size"][0, 1])
        w, h = self.w, self.h
        self._g0, self._k0 = _gbuffer_struct(g0, w, h)
        self._g1, self._k1 = _gbuffer_struct(g1, w, h) if g1 is not None else (None, None)
        self._s, self._ks = _scene_struct(scene)
        self.hdr32 = np.zeros((h, w, 4), np.float32)
        self.hdr16 = np.zeros((h, w, 4), np.uint16)
        # rows outside the sampled band come from `opaque_full16` when given (e.g. the GPU's opaque frame)
        self.levels = [np.zeros((h, w, 4), np.uint16) if opaque_full16 is None else np.array(opaque_full16, np.uint16, copy=True)]
        for _ in range(1, mip_levels_for_size(w, h)):
            sh, sw = self.levels[-1].shape[:2]
            self.levels.append(np.zeros((max(1, sh // 2), max(1, sw // 2), 4), np.uint16))
        self._pyr, self._kp = make_pyramid_struct(self.levels)
        self._lut, self._kl = make_lut_struct(lut_rgba8)
        self._tm = _c(tonemap_params, abi.baked_lottes_tonemapper_params)
        self.srgb8 = np.zeros((h, w, 4), np.uint8)

    def opaque(self, y0, y1):
        lib().orc_shade_opaque_frame(C.byref(self._g0), C.byref(self._s), C.c_uint32(y0), C.c_uint32(y1), _p(self.hdr32),
                                     _p(self.hdr16), _p(self.levels[0]))

    def mips(self):
        for l in range(1, len(self.levels)):
            src, dst = self.levels[l - 1], self.levels[l]
            lib().orc_downsample_level(_p(src), C.c_uint32(src.shape[1]), C.c_uint32(src.shape[0]), _p(dst),
                                       C.c_uint32(dst.shape[1]), C.c_uint32(dst.shape[0]))

    def transmission(self, y0, y1):
        if self._g1 is not None:
            lib().orc_shade_transmission_frame(C.byref(self._g1), C.byref(self._s), C.byref(self._pyr), C.byref(self._lut),
                                               C.c_uint32(y0), C.c_uint32(y1), _p(self.hdr32), _p(self.hdr16))

    def tonemap(self, y0, y1):
        lib().orc_tonemap_frame(_p(self.hdr16), C.c_uint32(self.w), C.c_uint32(self.h), C.c_uint32(y0), C.c_uint32(y1),
                                _p(self._tm), _p(self.srgb8))


# ---- vertex stage / alpha clip, exposed for the comparison with the reference's shipped modules --------------------
class _V2(C.Structure):
    _fields_ = [("x", C.c_float), ("y", C.c_float)]


class _V3(C.Structure):
    _fields_ = [("x", C.c_float), ("y", C.c_float), ("z", C.c_float)]


class _V4(C.Structure):
    _fields_ = [("x", C.c_float), ("y", C.c_float), ("z", C.c_float), ("w", C.c_float)]


def vertex_instanced_with_scale(positions, normals, uvs, instance_index, instances, push_constants):
    positions, normals = _c(positions, np.float32).reshape(-1, 3), _c(normals, np.float32).reshape(-1, 3)
    instances = _c(instances, abi.instance)
    pc = _c(push_constants, abi.push_constants)
    n = len(positions)
    out = dict(clip=np.zeros((n, 4), np.float32), position=np.zeros((n, 3), np.float32), normal=np.zeros((n, 3), np.float32),
               uv=_c(uvs, np.float32).reshape(-1, 2).copy(), material_id=np.zeros(n, np.uint32), scale=np.zeros(n, np.float32))
    L = lib()
    L.orc_vertex_instanced_with_scale.argtypes = [_V3, _V3, C.c_void_p, C.c_void_p] + [C.c_void_p] * 5
    L.orc_vertex_instanced_with_scale.restype = None
    isz = abi.instance.itemsize
    for i in range(n):
        L.orc_vertex_instanced_with_scale(_V3(*positions[i]), _V3(*normals[i]), instances.ctypes.data + isz * int(instance_index[i]),
                                          pc.ctypes.data, out["clip"].ctypes.data + 16 * i, out["position"].ctypes.data + 12 * i,
                                          out["normal"].ctypes.data + 12 * i, out["material_id"].ctypes.data + 4 * i,
                                          out["scale"].ctypes.data + 4 * i)
    return out


def alpha_clip(uvs, duv, material_id, scene):
    """depth_pre_pass_alpha_clip per fragment: 1 = discarded."""
    uvs = _c(uvs, np.float32).reshape(-1, 2)
    duv = _c(duv, np.float32).reshape(-1, 4) if duv is not None else np.zeros((len(uvs), 4), np.float32)
    s, ks = _scene_struct(scene)
    L = lib()
    L.orc_alpha_clip_kills.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, _V2, _V2, _V2]
    L.orc_alpha_clip_kills.restype = C.c_int
    msz = abi.material_info.itemsize
    out = np.zeros(len(uvs), np.uint8)
    for i in range(len(uvs)):
        out[i] = L.orc_alpha_clip_kills(ks.m.ctypes.data + msz * int(material_id[i]), s.textures, s.n_textures, _V2(*uvs[i]),
                                        _V2(*duv[i, :2]), _V2(*duv[i, 2:]))
    return out
