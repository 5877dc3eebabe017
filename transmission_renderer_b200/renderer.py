"""`Renderer`: Python mirror of the C ABI (include/tr_abi.h), one method per `tr_*` entry point.

It plays the part of the reference's frame recorder `record()` (src/main.rs:1551-2263) for
tests and benchmarks: same pass names, same argument structs, same error behaviour (a
non-zero status raises `TrError` carrying `tr_last_error()`, like `anyhow::Result` + `?`).
All arithmetic happens in libtr.so on the GPU.
"""
import ctypes as C

import numpy as np

from . import abi, host


def _lib():
    from . import lib
    return lib()


def _check(status):
    from . import _check as chk
    chk(status)


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _c(a, dtype):
    return np.ascontiguousarray(a, dtype=dtype)


def _device_rows(a, who, device, row_bytes, typestrs):
    """(pointer, rows) of a device array (a CUDA torch tensor, or any object with `__cuda_array_interface__`) holding rows of
    `row_bytes` bytes, or None when `a` is host data.  The array must be C-contiguous, of one of `typestrs` ('<f4': shape
    (n, row_bytes / 4); '|u1': shape (n, row_bytes) or (n * row_bytes,)), and on `device` when it says where it lives (torch's
    `.device.index`, CuPy's `.device.id`)."""
    cai = getattr(a, "__cuda_array_interface__", None)
    if cai is None:
        return None
    shape, typestr, strides = tuple(cai["shape"]), cai["typestr"], cai.get("strides")
    if typestr not in typestrs:
        raise TypeError(f"{who}: a device array of {typestr}; expected one of {', '.join(typestrs)}")
    item = int(typestr[2:])
    if typestr == "|u1" and len(shape) == 1 and shape[0] % row_bytes == 0:
        rows = shape[0] // row_bytes
    elif len(shape) == 2 and shape[1] * item == row_bytes:
        rows = shape[0]
    else:
        raise ValueError(f"{who}: device array of shape {shape} and type {typestr} is not rows of {row_bytes} bytes")
    if strides is not None and rows > 1 and tuple(strides) != tuple(item * int(np.prod(shape[k + 1:])) for k in range(len(shape))):
        raise ValueError(f"{who}: the device array is not C-contiguous (strides {strides})")
    dev = getattr(a, "device", None)
    where = getattr(dev, "index", None)
    if where is None:
        where = getattr(dev, "id", None)
    if where is not None and int(where) != device:
        raise ValueError(f"{who}: the device array is on device {where}, the renderer on device {device}")
    return (cai["data"][0] if rows else None), rows


class _Config(C.Structure):
    _fields_ = [("width", C.c_uint32), ("height", C.c_uint32), ("device", C.c_int32), ("band_y0", C.c_uint32),
                ("band_y1", C.c_uint32), ("flags", C.c_uint32)]


class _Planes(C.Structure):
    _fields_ = [("depth", C.c_void_p), ("normal", C.c_void_p), ("uv", C.c_void_p), ("material_id", C.c_void_p),
                ("scale", C.c_void_p), ("position", C.c_void_p), ("duv", C.c_void_p), ("ddepth", C.c_void_p)]


_PLANES = ("depth", "normal", "uv", "material_id", "scale", "position", "duv", "ddepth")


class Renderer:
    def __init__(self, width, height, device=0, band=None, f32_debug=False):
        self._ctx = C.c_void_p()
        self.width, self.height = int(width), int(height)
        y0, y1 = band if band is not None else (0, 0)
        cfg = _Config(self.width, self.height, device, y0, y1, abi.TR_FLAG_HDR_F32_DEBUG if f32_debug else 0)
        _check(_lib().tr_create(C.byref(cfg), C.byref(self._ctx)))
        self.f32_debug = f32_debug
        self.device = int(device)
        self.acceleration_structure_address = 0   # the handle of the last build_acceleration_structures (RendererGroup.frame)
        self._keep = []

    # -- lifecycle -------------------------------------------------------------------
    def close(self):
        if self._ctx:
            _check(_lib().tr_destroy(self._ctx))   # refused while the context is a member of a RendererGroup
            self._ctx = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def resize(self, width, height):
        _check(_lib().tr_resize(self._ctx, C.c_uint32(width), C.c_uint32(height)))
        self.width, self.height = int(width), int(height)

    def set_band(self, y0, y1):
        _check(_lib().tr_set_band(self._ctx, C.c_uint32(y0), C.c_uint32(y1)))

    def set_stream(self, cuda_stream_handle):
        _check(_lib().tr_set_stream(self._ctx, C.c_void_p(cuda_stream_handle)))

    def sync(self):
        _check(_lib().tr_sync(self._ctx))

    # -- uploads ------------------------------------------------------------------------
    def set_instances(self, instances):
        a = _c(instances, abi.instance)
        _check(_lib().tr_set_instances(self._ctx, _p(a), C.c_uint32(len(a))))

    def update_instance_transforms(self, transforms, first=0):
        """New transforms (the 32-byte packed similarity: translation_and_scale, rotation) for instances [first, first + n);
        their primitive and material ids stay.  Stream-ordered; with ray queries, update the top level before the next
        frame.  `transforms`: host data as (n, 8) float32, or a device array (a CUDA tensor or any object with
        `__cuda_array_interface__`, on this renderer's device) of (n, 8) float32, (n, 32) uint8 or (n * 32,) uint8, read in
        stream order on the context stream (order its producer before the call)."""
        dev = _device_rows(transforms, "update_instance_transforms", self.device, 32, ("<f4", "|u1"))
        if dev is not None:
            ptr, n = dev
        else:
            a = _c(transforms, np.float32).reshape(-1, 8)
            ptr, n = (a.ctypes.data if len(a) else None), len(a)
        _check(_lib().tr_update_instance_transforms(self._ctx, C.c_uint32(first), C.c_uint32(n), C.c_void_p(ptr)))

    def set_primitives(self, primitives):
        a = _c(primitives, abi.primitive_info)
        _check(_lib().tr_set_primitives(self._ctx, _p(a), C.c_uint32(len(a))))

    def set_materials(self, materials):
        a = _c(materials, abi.material_info)
        _check(_lib().tr_set_materials(self._ctx, _p(a), C.c_uint32(len(a))))

    def set_lights(self, lights):
        """`lights`: abi.light records on the host, or a device array of their bytes (a CUDA tensor or any object with
        `__cuda_array_interface__`, on this renderer's device): (n, 12) float32, (n, 48) uint8 or (n * 48,) uint8, copied in
        stream order on the context stream (order its producer before the call)."""
        dev = _device_rows(lights, "set_lights", self.device, abi.light.itemsize, ("<f4", "|u1"))
        if dev is not None:
            ptr, n = dev
            _check(_lib().tr_set_lights(self._ctx, C.c_void_p(ptr), C.c_uint32(n)))
            return
        a = _c(lights, abi.light)
        _check(_lib().tr_set_lights(self._ctx, _p(a) if len(a) else None, C.c_uint32(len(a))))

    def set_uniforms(self, uniforms):
        a = _c(uniforms, abi.uniforms)
        _check(_lib().tr_set_uniforms(self._ctx, _p(a)))

    def set_ggx_lut(self, rgba8):
        a = _c(rgba8, np.uint8)
        _check(_lib().tr_set_ggx_lut(self._ctx, _p(a), C.c_uint32(a.shape[1]), C.c_uint32(a.shape[0])))

    def set_texture(self, index, levels, srgb):
        """levels: list of (h, w, 4) uint8 mips, level 0 first (scenes.make_mips)."""
        lv = [_c(l, np.uint8) for l in levels]
        ptrs = (C.c_void_p * len(lv))(*[l.ctypes.data for l in lv])
        _check(_lib().tr_set_texture(self._ctx, C.c_uint32(index), ptrs, C.c_uint32(len(lv)), C.c_uint32(lv[0].shape[1]),
                                     C.c_uint32(lv[0].shape[0]), C.c_int32(1 if srgb else 0)))

    def set_texture_async(self, index, rgba8, srgb, n_levels=0):
        """rgba8: (h, w, 4) uint8, level 0 only; levels 1 .. n_levels - 1 (0: the full chain) are built on the device in
        stream order, bit-equal to set_texture(scenes.make_mips(rgba8, srgb)).  A page-locked array is read in stream order
        (keep it alive and unchanged until the stream has passed the call); a pageable one is copied during the call."""
        a = np.asarray(rgba8)
        if a.dtype != np.uint8 or a.ndim != 3 or a.shape[2] != 4 or not a.flags.c_contiguous:
            a = _c(a, np.uint8).reshape(a.shape[0], a.shape[1], 4)
        _check(_lib().tr_set_texture_async(self._ctx, C.c_uint32(index), _p(a), C.c_uint32(a.shape[1]), C.c_uint32(a.shape[0]),
                                           C.c_int32(1 if srgb else 0), C.c_uint32(n_levels)))

    def read_texture_level(self, index, level):
        """(h, w, 4) float32: level `level` of image `index` as the samplers read it (decoded to linear)."""
        w, h = C.c_uint32(0), C.c_uint32(0)
        _check(_lib().tr_read_texture_level(self._ctx, C.c_uint32(index), C.c_uint32(level), None, C.byref(w), C.byref(h)))
        a = np.zeros((h.value, w.value, 4), np.float32)
        _check(_lib().tr_read_texture_level(self._ctx, C.c_uint32(index), C.c_uint32(level), _p(a), C.byref(w), C.byref(h)))
        return a

    def set_textures(self, textures, on_device=False):
        """on_device: bind only each levels[0] (set_texture_async) and let the device build the chains."""
        for i, t in enumerate(textures):
            if on_device:
                self.set_texture_async(i, t["levels"][0], t["srgb"])
            else:
                self.set_texture(i, t["levels"], t["srgb"])

    def set_mesh(self, positions, normals, uvs, indices):
        p, n, u, i = _c(positions, np.float32), _c(normals, np.float32), _c(uvs, np.float32), _c(indices, np.uint32)
        _check(_lib().tr_set_mesh(self._ctx, _p(p), _p(n), _p(u), C.c_uint32(len(p)), _p(i), C.c_uint32(i.size)))

    def update_mesh_vertices(self, positions, normals, first_vertex=0):
        """New positions and normals ((n, 3) float32 each) for vertices [first_vertex, first_vertex + n) of the mesh, in
        stream order: the culling spheres and, once built, the bottom-level acceleration structures follow on the device.
        After it, a traced frame needs a top-level update first.  Page-locked arrays are read in stream order.  Either
        array may instead be a device array ((n, 3) float32, C-contiguous, on this renderer's device: a CUDA tensor or any
        object with `__cuda_array_interface__`), read in stream order on the context stream (order its producer before the
        call); host and device arrays may be mixed."""
        ptrs, counts, keep = [], [], []
        for a in (positions, normals):
            dev = _device_rows(a, "update_mesh_vertices", self.device, 12, ("<f4",))
            if dev is None:
                h = _c(a, np.float32).reshape(-1, 3)
                keep.append(h)
                dev = (h.ctypes.data if len(h) else None), len(h)
            ptrs.append(C.c_void_p(dev[0]))
            counts.append(dev[1])
        if counts[0] != counts[1]:
            raise ValueError(f"update_mesh_vertices: {counts[0]} positions but {counts[1]} normals")
        _check(_lib().tr_update_mesh_vertices(self._ctx, C.c_uint32(first_vertex), C.c_uint32(counts[0]), *ptrs))

    def read_chunk_spheres(self):
        """(n, 4) float32: the binning pass's culling spheres (object-space centre, radius), one per 64 consecutive
        triangles of every primitive, primitive after primitive."""
        n = C.c_uint32(0)
        _check(_lib().tr_read_chunk_spheres(self._ctx, None, C.c_uint32(0), C.byref(n)))
        out = np.zeros((n.value, 4), np.float32)
        _check(_lib().tr_read_chunk_spheres(self._ctx, _p(out) if len(out) else None, C.c_uint32(len(out)), C.byref(n)))
        return out

    # -- ray-queried shadows (`--ray-tracing`, src/main.rs:577-658) ---------------------------
    def build_acceleration_structures(self):
        """Bottom-level structures of every primitive + the top level over the instances with draw_buffer_index < 2.
        Returns the handle to put into PushConstants.acceleration_structure_address (src/main.rs:856-859)."""
        a = C.c_uint64(0)
        _check(_lib().tr_build_acceleration_structures(self._ctx, C.byref(a)))
        self.acceleration_structure_address = a.value
        return a.value

    def build_acceleration_structures_async(self):
        """The same structures built on the device in stream order: returns the handle without waiting for the GPU and
        reads the mesh and instances as the stream sees them (also the rebuild after update_mesh_vertices refits)."""
        a = C.c_uint64(0)
        _check(_lib().tr_build_acceleration_structures_async(self._ctx, C.byref(a)))
        self.acceleration_structure_address = a.value
        return a.value

    def update_top_level_acceleration_structure(self):
        a = C.c_uint64(0)
        _check(_lib().tr_update_top_level_acceleration_structure(self._ctx, C.byref(a)))
        self.acceleration_structure_address = a.value
        return a.value

    def update_top_level_acceleration_structure_async(self):
        """The same update built on the device in stream order: returns without waiting for the GPU; the next frame
        traces against it."""
        a = C.c_uint64(0)
        _check(_lib().tr_update_top_level_acceleration_structure_async(self._ctx, C.byref(a)))
        self.acceleration_structure_address = a.value
        return a.value

    def read_top_level_acceleration_structure(self):
        """(nodes, instances): the top level as built, abi.accel_node (node 0 is the root) and abi.accel_instance in
        leaf order."""
        nn, ni = C.c_uint32(0), C.c_uint32(0)
        _check(_lib().tr_read_top_level_acceleration_structure(self._ctx, None, C.c_uint32(0), C.byref(nn), None, C.c_uint32(0),
                                                                C.byref(ni)))
        nodes = np.zeros(nn.value, dtype=abi.accel_node)
        inst = np.zeros(ni.value, dtype=abi.accel_instance)
        _check(_lib().tr_read_top_level_acceleration_structure(self._ctx, _p(nodes), C.c_uint32(len(nodes)), C.byref(nn),
                                                                _p(inst) if len(inst) else None, C.c_uint32(len(inst)), C.byref(ni)))
        return nodes, inst

    def read_bottom_level_acceleration_structure(self):
        """(nodes, tris): every primitive's tree, abi.accel_node, one after the other in primitive order (each root first),
        and the triangles in leaf order, (n, 3, 4) float32 (x, y, z, 0); leaf references count from the primitive's first
        triangle."""
        nn, nt = C.c_uint32(0), C.c_uint32(0)
        _check(_lib().tr_read_bottom_level_acceleration_structures(self._ctx, None, C.c_uint32(0), C.byref(nn), None, C.c_uint32(0),
                                                                    C.byref(nt)))
        nodes = np.zeros(nn.value, dtype=abi.accel_node)
        tris = np.zeros((nt.value, 3, 4), np.float32)
        _check(_lib().tr_read_bottom_level_acceleration_structures(self._ctx, _p(nodes) if len(nodes) else None, C.c_uint32(len(nodes)),
                                                                    C.byref(nn), _p(tris) if len(tris) else None, C.c_uint32(len(tris)),
                                                                    C.byref(nt)))
        return nodes, tris

    def trace_shadow_rays(self, origins, directions, t_max):
        """(n,3), (n,3), (n,) -> (n,) uint8: 1 = lit, 0 = occluded (trace_shadow_ray, lighting.rs:97-125)."""
        o, d = _c(origins, np.float32).reshape(-1, 3), _c(directions, np.float32).reshape(-1, 3)
        t = _c(t_max, np.float32).reshape(-1)
        out = np.zeros(len(o), np.uint8)
        _check(_lib().tr_trace_shadow_rays(self._ctx, C.c_uint32(len(o)), _p(o), _p(d), _p(t), _p(out)))
        return out

    def read_shadow_mask(self, layer):
        """(5, h, w) uint32 occluded-ray bits of the last shading pass of `layer` (band rows)."""
        out = np.zeros((5, self.height, self.width), np.uint32)
        _check(_lib().tr_read_shadow_mask(self._ctx, C.c_int32(layer), _p(out)))
        return out

    # -- passes, in record() order --------------------------------------------------------
    def cull(self, culling_pc):
        _check(_lib().tr_cull(self._ctx, _p(_c(culling_pc, abi.culling_push_constants))))

    def build_clusters(self, wc_pc):
        _check(_lib().tr_build_clusters(self._ctx, _p(_c(wc_pc, abi.write_cluster_data_push_constants))))

    def assign_lights(self, al_pc):
        _check(_lib().tr_assign_lights(self._ctx, _p(_c(al_pc, abi.assign_lights_push_constants))))

    def visibility(self, pc):
        _check(_lib().tr_visibility(self._ctx, _p(_c(pc, abi.push_constants))))

    def shade_opaque(self, pc):
        _check(_lib().tr_shade_opaque(self._ctx, _p(_c(pc, abi.push_constants))))

    def allgather_opaque(self):
        _check(_lib().tr_allgather_opaque(self._ctx))

    def generate_mips(self):
        _check(_lib().tr_generate_mips(self._ctx))

    def shade_transmission(self, pc):
        _check(_lib().tr_shade_transmission(self._ctx, _p(_c(pc, abi.push_constants))))

    def tonemap(self, params):
        _check(_lib().tr_tonemap(self._ctx, _p(_c(params, abi.baked_lottes_tonemapper_params))))

    def frame(self, frame_params):
        _check(_lib().tr_frame(self._ctx, _p(_c(frame_params, abi.frame_params))))

    def begin_frame(self):
        """Start of a frame for the per-pass timers when the passes are called one by one (tr_frame does it itself)."""
        _check(_lib().tr_begin_frame(self._ctx))

    def enable_timing(self, on=True):
        _check(_lib().tr_enable_timing(self._ctx, C.c_int32(1 if on else 0)))

    def frame_times(self):
        t = np.zeros(1, dtype=abi.frame_times)
        _check(_lib().tr_read_frame_times(self._ctx, _p(t)))
        return {k: float(t[k][0]) for k in t.dtype.names}

    def pass_totals(self):
        """(sum of per-pass ms over the frames since enable_timing / the last call, number of frames)."""
        t = np.zeros(1, dtype=abi.frame_times)
        n = C.c_uint32(0)
        _check(_lib().tr_read_pass_totals(self._ctx, _p(t), C.byref(n)))
        return {k: float(t[k][0]) for k in t.dtype.names}, n.value

    # -- parity hooks ------------------------------------------------------------------------
    def set_gbuffer(self, layer, gbuffer):
        npx = self.width * self.height
        keep = dict(depth=_c(gbuffer["depth"], np.float32), normal=_c(gbuffer["normal"], np.float32),
                    material_id=_c(gbuffer["material_id"], np.uint32))
        assert keep["depth"].size == npx and keep["normal"].size == npx * 3 and keep["material_id"].size == npx
        for k, dt, mult in (("uv", np.float32, 2), ("scale", np.float32, 1), ("position", np.float32, 3),
                            ("duv", np.float32, 4), ("ddepth", np.float32, 2)):
            v = gbuffer.get(k)
            keep[k] = None if v is None else _c(v, dt)
            assert keep[k] is None or keep[k].size == npx * mult
        planes = _Planes(*[None if keep[k] is None else keep[k].ctypes.data for k in _PLANES])
        _check(_lib().tr_set_gbuffer(self._ctx, C.c_int32(layer), C.byref(planes)))
        self.sync()

    def read_gbuffer(self, layer, with_position=False, derivatives=False):
        h, w = self.height, self.width
        g = dict(depth=np.zeros((h, w), np.float32), normal=np.zeros((h, w, 3), np.float32),
                 uv=np.zeros((h, w, 2), np.float32), material_id=np.zeros((h, w), np.uint32),
                 scale=np.zeros((h, w), np.float32), position=np.zeros((h, w, 3), np.float32) if with_position else None,
                 duv=np.zeros((h, w, 4), np.float32) if derivatives else None,
                 ddepth=np.zeros((h, w, 2), np.float32) if derivatives else None)
        planes = _Planes(*[None if g[k] is None else g[k].ctypes.data for k in _PLANES])
        _check(_lib().tr_read_gbuffer(self._ctx, C.c_int32(layer), C.byref(planes)))
        return g

    def set_opaque_frame(self, rgba16f_bits):
        a = _c(rgba16f_bits, np.uint16)
        assert a.size == self.width * self.height * 4
        _check(_lib().tr_set_opaque_frame(self._ctx, _p(a)))
        self.sync()

    def set_hdr(self, rgba16f_bits):
        a = _c(rgba16f_bits, np.uint16)
        assert a.size == self.width * self.height * 4
        _check(_lib().tr_set_hdr(self._ctx, _p(a)))
        self.sync()

    def set_cluster_lights(self, counts, indices):
        a, b = _c(counts, np.uint32), _c(indices, np.uint32)
        _check(_lib().tr_set_cluster_lights(self._ctx, _p(a), _p(b)))
        self.sync()

    def read_visible_instances(self):
        n = C.c_uint32(0)
        _check(_lib().tr_read_visible_instances(self._ctx, None, C.c_uint32(0), C.byref(n)))
        ids = np.zeros(max(1, n.value), dtype=np.uint32)
        _check(_lib().tr_read_visible_instances(self._ctx, _p(ids), C.c_uint32(len(ids)), C.byref(n)))
        return ids[: n.value].copy()

    def read_instance_counts(self, n_primitives):
        a = np.zeros(n_primitives, dtype=np.uint32)
        _check(_lib().tr_read_instance_counts(self._ctx, _p(a), C.c_uint32(n_primitives)))
        return a

    def read_draws(self, bucket):
        n = C.c_uint32(0)
        _check(_lib().tr_read_draws(self._ctx, C.c_uint32(bucket), None, C.c_uint32(0), C.byref(n)))
        cmds = np.zeros(max(1, n.value), dtype=abi.draw_indexed_indirect_command)
        _check(_lib().tr_read_draws(self._ctx, C.c_uint32(bucket), _p(cmds), C.c_uint32(len(cmds)), C.byref(n)))
        return cmds[: n.value].copy()

    def read_cluster_aabbs(self, n_clusters):
        a = np.zeros(n_clusters, dtype=abi.cluster_aabb)
        _check(_lib().tr_read_cluster_aabbs(self._ctx, _p(a), C.c_uint32(n_clusters)))
        return a

    def read_cluster_lights(self, n_clusters):
        counts = np.zeros(n_clusters, dtype=np.uint32)
        indices = np.zeros(n_clusters * abi.TR_MAX_LIGHTS_PER_CLUSTER, dtype=np.uint32)
        _check(_lib().tr_read_cluster_lights(self._ctx, _p(counts), _p(indices)))
        return counts, indices

    def read_hdr(self):
        a = np.zeros((self.height, self.width, 4), dtype=np.uint16)
        _check(_lib().tr_read_hdr(self._ctx, _p(a)))
        return a

    def read_hdr_f32(self):
        a = np.zeros((self.height, self.width, 4), dtype=np.float32)
        _check(_lib().tr_read_hdr_f32(self._ctx, _p(a)))
        return a

    def mip_levels(self):
        n = C.c_uint32(0)
        _check(_lib().tr_mip_levels(self._ctx, C.byref(n)))
        return n.value

    def read_pyramid_level(self, level):
        w, h = C.c_uint32(0), C.c_uint32(0)
        _check(_lib().tr_read_pyramid_level(self._ctx, C.c_uint32(level), None, C.byref(w), C.byref(h)))
        a = np.zeros((h.value, w.value, 4), dtype=np.uint16)
        _check(_lib().tr_read_pyramid_level(self._ctx, C.c_uint32(level), _p(a), C.byref(w), C.byref(h)))
        return a

    def read_srgb8(self, out=None):
        a = np.zeros((self.height, self.width, 4), dtype=np.uint8) if out is None else out
        _check(_lib().tr_read_srgb8(self._ctx, _p(a)))
        return a

    # -- glam-pbr contracts --------------------------------------------------------------------
    def read_srgb8_async(self, out):
        """Enqueue the band read-back behind the frame just recorded; `out` (H, W, 4) uint8, ideally pinned."""
        assert out.dtype == np.uint8 and out.size == self.width * self.height * 4 and out.flags.c_contiguous
        _check(_lib().tr_read_srgb8_async(self._ctx, _p(out)))

    def wait_readback(self):
        _check(_lib().tr_wait_readback(self._ctx))

    def eval_basic_brdf(self, params):
        a = _c(params, abi.basic_brdf_params)
        out = np.zeros(len(a), dtype=abi.brdf_result)
        _check(_lib().tr_eval_basic_brdf(self._ctx, C.c_uint32(len(a)), _p(a), _p(out)))
        return out

    def eval_transmission_btdf(self, params):
        a = _c(params, abi.transmission_btdf_params)
        out = np.zeros((len(a), 3), dtype=np.float32)
        _check(_lib().tr_eval_transmission_btdf(self._ctx, C.c_uint32(len(a)), _p(a), _p(out)))
        return out

    def eval_point_light(self, params):
        """The frame kernels' light loop for one (pixel, point light) pair per element."""
        a = _c(params, abi.point_light_params)
        out = np.zeros(len(a), dtype=abi.point_light_result)
        _check(_lib().tr_eval_point_light(self._ctx, C.c_uint32(len(a)), _p(a), _p(out)))
        return out

    def eval_ibl_volume_refraction(self, proj_view, params):
        a = _c(params, abi.ibl_volume_refraction_params)
        pv = _c(np.asarray(proj_view, dtype=np.float32).T, np.float32)
        out = np.zeros((len(a), 3), dtype=np.float32)
        _check(_lib().tr_eval_ibl_volume_refraction(self._ctx, C.c_uint32(len(a)), _p(pv), _p(a), _p(out)))
        return out

    # -- multi-GPU ---------------------------------------------------------------------------------
    @staticmethod
    def comm_unique_id():
        buf = (C.c_uint8 * 128)()
        _check(_lib().tr_comm_unique_id(buf))
        return bytes(buf)

    def comm_init(self, unique_id, rank, n_ranks):
        buf = (C.c_uint8 * 128).from_buffer_copy(unique_id)
        _check(_lib().tr_comm_init(self._ctx, buf, C.c_int32(rank), C.c_int32(n_ranks)))

    def set_bands(self, bounds):
        """n_ranks + 1 ascending row boundaries, the same on every rank (tr_set_bands)."""
        a = _c(bounds, np.uint32)
        _check(_lib().tr_set_bands(self._ctx, _p(a), C.c_uint32(len(a))))

    def comm_destroy(self):
        _check(_lib().tr_comm_destroy(self._ctx))

    def peer_export(self):
        buf = (C.c_uint8 * 64)()
        _check(_lib().tr_peer_export(self._ctx, buf))
        return bytes(buf)

    def peer_attach(self, rank, n_ranks, handles):
        blob = b"".join(handles)
        buf = (C.c_uint8 * len(blob)).from_buffer_copy(blob)
        _check(_lib().tr_peer_attach(self._ctx, C.c_int32(rank), C.c_int32(n_ranks), buf))

    def device_buffer(self, what):
        ptr, nbytes = C.c_void_p(), C.c_size_t(0)
        _check(_lib().tr_device_buffer(self._ctx, C.c_int32(what), C.byref(ptr), C.byref(nbytes)))
        return ptr.value, nbytes.value

    # -- diagnostics -----------------------------------------------------------------------------------
    @staticmethod
    def launch_count():
        n = C.c_uint64(0)
        _check(_lib().tr_launch_count(C.byref(n)))
        return n.value

    def raster_stats(self, reset=True):
        out = (C.c_uint64 * 4)()
        _check(_lib().tr_raster_stats(self._ctx, out, C.c_int32(1 if reset else 0)))
        return dict(box_pixels=out[0], box_pixels_after_hiz=out[1], exact_evaluations=out[2], span_pixels=out[3])

    def measure_fp32_peak(self):
        v = C.c_float(0)
        _check(_lib().tr_measure_fp32_peak(self._ctx, C.byref(v)))
        return v.value

    def measure_hbm_copy(self):
        v = C.c_float(0)
        _check(_lib().tr_measure_hbm_copy(self._ctx, C.byref(v)))
        return v.value


_BAND_PASSES = ("visibility_ms", "shade_opaque_ms", "shade_transmission_ms", "tonemap_ms")   # a band's own cost (parallel.py)


class RendererGroup:
    """Several `Renderer`s of this thread rendering the bands of ONE frame (tr_group_*): member k renders band k, and its
    opaque pass stores the band into every member's opaque frame directly.  The members may sit on different devices or on
    the same one.  The reference's host is one thread with one queue (src/main.rs:243); this is how such a host drives
    several GPUs.

        with Renderer(w, h, device=0) as a, Renderer(w, h, device=1) as b, RendererGroup([a, b]) as g:
            g.frame(camera.frame_params())
            image = g.read_srgb8()

    While the group lives, the members' frame-wide calls (frame, shade_opaque, resize, set_band(s), close ...) raise;
    uploads, build_acceleration_structures, timers and reads stay per member."""

    def __init__(self, renderers):
        self.renderers = list(renderers)
        n = len(self.renderers)
        ctxs = (C.c_void_p * max(n, 1))(*[r._ctx.value for r in self.renderers])
        self._g = C.c_void_p()
        _check(_lib().tr_group_create(ctxs, C.c_uint32(n), C.byref(self._g)))
        self.width, self.height = self.renderers[0].width, self.renderers[0].height
        self.bounds = self._equal_bounds()

    def _equal_bounds(self):
        n = len(self.renderers)
        return [host.band_rows(self.height, k, n)[0] for k in range(n)] + [self.height]

    # -- lifecycle ---------------------------------------------------------------------------------
    def close(self):
        """tr_group_destroy: waits for every member, which renders the whole frame again."""
        if self._g:
            st = _lib().tr_group_destroy(self._g)
            self._g = C.c_void_p()
            _check(st)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # -- frame -----------------------------------------------------------------------------------------
    def set_bands(self, bounds):
        """n + 1 ascending row boundaries, 0 ... height; member k renders rows [bounds[k], bounds[k+1])."""
        a = _c(bounds, np.uint32)
        _check(_lib().tr_group_set_bands(self._g, _p(a), C.c_uint32(len(a))))
        self.bounds = [int(v) for v in a]

    def resize(self, width, height):
        """Every member at the new size; the bands return to equal rows."""
        _check(_lib().tr_group_resize(self._g, C.c_uint32(width), C.c_uint32(height)))
        for r in self.renderers:
            r.width, r.height = int(width), int(height)
        self.width, self.height = int(width), int(height)
        self.bounds = self._equal_bounds()

    def frame(self, params):
        """One frame across the members.  `params`: one frame-params struct for all of them, or a list of one per member.
        A single struct with ray queries on (acceleration_structure_address != 0) gets each member's own handle."""
        n = len(self.renderers)
        if isinstance(params, (list, tuple)):
            if len(params) != n:
                raise ValueError(f"{len(params)} frame params for {n} members")
            p = np.zeros(n, dtype=abi.frame_params)   # not np.concatenate: it packs the struct, dropping the ABI's padding
            for k, q in enumerate(params):
                p[k] = _c(q, abi.frame_params).reshape(-1)[0]
        else:
            one = _c(params, abi.frame_params).reshape(-1)
            if len(one) != 1:
                raise ValueError("frame(params): one struct, or a list of one per member")
            p = np.repeat(one, n)
            if one["push_constants"]["acceleration_structure_address"][0] != 0:
                for k, r in enumerate(self.renderers):
                    p[k]["push_constants"]["acceleration_structure_address"] = r.acceleration_structure_address
        _check(_lib().tr_group_frame(self._g, _p(p)))

    def sync(self):
        _check(_lib().tr_group_sync(self._g))

    # -- scene -------------------------------------------------------------------------------------------
    def replicate_scene(self, source=0):
        """Copies member `source`'s scene (everything its uploads and builds made, as its stream sees it now) into every
        other member, GPU to GPU in stream order, without waiting for the device unless a buffer grows: load one member,
        then replicate.  Returns every member's acceleration-structure handle (0 where the source has no valid top level),
        which also becomes each member's `acceleration_structure_address`."""
        n = len(self.renderers)
        out = (C.c_uint64 * n)()
        _check(_lib().tr_group_replicate_scene(self._g, C.c_uint32(source), out))
        for r, a in zip(self.renderers, out):
            r.acceleration_structure_address = int(a)
        return [int(a) for a in out]

    # -- whole-frame reads ---------------------------------------------------------------------------
    def read_srgb8(self, out=None):
        a = np.zeros((self.height, self.width, 4), dtype=np.uint8) if out is None else out
        assert a.dtype == np.uint8 and a.size == self.width * self.height * 4 and a.flags.c_contiguous
        _check(_lib().tr_group_read_srgb8(self._g, _p(a)))
        return a

    def read_hdr(self):
        """The RGBA16F frame stitched from every member's band."""
        out = np.zeros((self.height, self.width, 4), dtype=np.uint16)
        for k, r in enumerate(self.renderers):
            y0, y1 = self.bounds[k], self.bounds[k + 1]
            out[y0:y1] = r.read_hdr()[y0:y1]
        return out

    def pass_totals(self):
        """Every member's (per-pass ms summed over the frames since its timers were switched on, number of frames)."""
        return [r.pass_totals() for r in self.renderers]

    def balance_bands(self, run_frames, iterations=4):
        """Move the band boundaries until every member's band costs about the same: the in-process form of
        parallel.balance_bands, with the same cost model (parallel.balanced_bounds).  `run_frames()` renders a few group
        frames.  Returns the final boundaries."""
        from . import parallel
        bounds = list(self.bounds)
        if len(self.renderers) == 1:
            return bounds
        for _ in range(iterations):
            run_frames()             # untimed: the first frames after new boundaries grow buffers
            self.sync()
            for r in self.renderers:
                r.enable_timing(True)
            run_frames()
            self.sync()
            cost = []
            for r in self.renderers:
                totals, n = r.pass_totals()
                r.enable_timing(False)
                cost.append(sum(totals[k] for k in _BAND_PASSES) / max(n, 1))
            bounds = parallel.balanced_bounds(bounds, cost)
            self.set_bands(bounds)
        return bounds
