"""Device sources: tr_update_mesh_vertices and tr_set_lights fed from device memory, and tr_update_instance_transforms (new
transforms for a range of instances, ids kept) fed from host or device memory.  A device-sourced sequence must render byte for
byte what the host-sourced one renders, read its source in stream order on the context stream, never wait for the device,
and let the later of two light uploads before one frame win, whichever path each took."""
import ctypes as C
import time

import numpy as np
import pytest

from accel_checks import _deform, _hold, _pinned, _records_key, _upload_scene
from transmission_renderer_b200 import Renderer, RendererGroup, TrError, abi, host, lib, scenes

pytestmark = pytest.mark.gpu
f32 = np.float32
TR_ERR_INVALID_ARG, TR_ERR_STATE = -1, -6


# ---------------------------------------------------------------------------------------------------------- helpers
def _dev(a):
    """A CUDA tensor with the bytes of `a`: float32 arrays keep their shape, records become (n * itemsize,) uint8."""
    import torch
    a = np.ascontiguousarray(a)
    t = torch.from_numpy(a if a.dtype == f32 else a.view(np.uint8).reshape(-1))
    return t.cuda()


def _transforms(inst):
    """(n, 8) float32: the packed similarity of every instance record (translation_and_scale, rotation)."""
    return np.ascontiguousarray(np.concatenate([inst["translation_and_scale"], inst["rotation"]], 1), f32)


def _rotated(instances, f, first=0, last=None):
    """The instances with [first, last) turned about a tilted axis by 0.05 (f + 1) rad and nudged sideways (the records)."""
    last = len(instances) if last is None else last
    out = instances.copy()
    ang = 0.05 * (f + 1)
    ax = np.array([0.3, 1.0, 0.2]) / np.linalg.norm([0.3, 1.0, 0.2])
    x1, y1, z1, w1 = *(ax * np.sin(ang / 2)), np.cos(ang / 2)
    x2, y2, z2, w2 = instances["rotation"][first:last].astype(np.float64).T
    out["rotation"][first:last] = np.stack([w1 * x2 + x1 * w2 + y1 * z2 - z1 * y2, w1 * y2 - x1 * z2 + y1 * w2 + z1 * x2,
                                            w1 * z2 + x1 * y2 - y1 * x2 + z1 * w2, w1 * w2 - x1 * x2 - y1 * y2 - z1 * z2], 1)
    out["translation_and_scale"][first:last, 0] += f32(0.1 * np.sin(f + 1.0))
    return out


def _lights(s, k):
    """Version k of the scene's lights: emission scaled, positions shifted, every third light dropped for odd k."""
    lights = s["lights"].copy()
    lights["colour_emission_and_falloff_distance_sq"][:, :3] *= f32(1.0 + 0.4 * k)
    lights["position_and_spotlight_epsilon"][:, 0] += f32(0.3 * k)
    if k % 2:
        lights = lights[np.arange(len(lights)) % 3 != 2]
    return np.ascontiguousarray(lights).astype(abi.light)


def _n_clusters(s):
    u = s["uniforms"]
    return int(u["num_clusters"].reshape(-1)[0]) * int(u["num_clusters"].reshape(-1)[1]) * int(u["num_depth_slices"].reshape(-1)[0])


def _sync_torch():
    import torch
    torch.cuda.synchronize()


def _frame_outputs(r, rq):
    out = {"hdr": r.read_hdr(), "srgb8": r.read_srgb8()}
    for layer in (0, 1):
        g = r.read_gbuffer(layer)
        for name in ("depth", "normal", "uv", "material_id", "scale"):
            out[f"layer {layer} {name}"] = g[name]
        if rq:
            out[f"layer {layer} shadow mask"] = r.read_shadow_mask(layer)
    return out


def _assert_equal(got, want, what):
    for name in want:
        assert got[name].tobytes() == want[name].tobytes(), f"{what}: {name} differs"


# ---------------------------------------------------------------------------------------------------------- 1. vertices
@pytest.mark.parametrize("rq", [False, True], ids=["rq_off", "rq_on"])
def test_vertex_updates_equal_host(ggx_lut, rq):
    """Deforming updates (whole mesh, partial ranges, device positions with host normals) from device memory against the
    same updates from host memory: chunk spheres, bottom-level trees, G-buffer planes, shadow masks, fp16 HDR and sRGB8."""
    w, h = 480, 270
    s = scenes.shadow_scene(w, h)
    cam, tm = s["camera"], host.default_tonemap_params()
    nv = len(s["mesh"]["positions"])
    steps = [(0, nv), (100, nv // 2), (nv // 3, nv - 7), (0, nv)]
    mesh, poses = s["mesh"], []
    for k, (a, b) in enumerate(steps):
        pos, nrm, mesh = _deform(mesh, k + 1, a, b, amp=0.06)
        poses.append((a, pos, nrm, _dev(pos), _dev(nrm)))
    _sync_torch()
    ctx = [Renderer(w, h), Renderer(w, h)]
    try:
        handles = []
        for r in ctx:
            _upload_scene(r, ggx_lut, s)
            handles.append(r.build_acceleration_structures() if rq else 0)
            r.frame(cam.frame_params(tm, acceleration_structure_address=handles[-1]))
        for k, (a, pos, nrm, dpos, dnrm) in enumerate(poses):
            ctx[0].update_mesh_vertices(pos, nrm, first_vertex=a)
            # step 2 mixes the kinds: device positions, host normals
            ctx[1].update_mesh_vertices(dpos, nrm if k == 2 else dnrm, first_vertex=a)
            outs = []
            for r, hdl in zip(ctx, handles):
                if rq:
                    assert r.update_top_level_acceleration_structure_async() == hdl
                r.frame(cam.frame_params(tm, acceleration_structure_address=hdl))
                o = _frame_outputs(r, rq)
                o["chunk spheres"] = r.read_chunk_spheres()
                if rq:   # a refitted box may carry either sign of a zero (arrival order): compared with +0 for -0
                    nodes, o["bottom-level triangles"] = r.read_bottom_level_acceleration_structure()
                    for name in ("lo0", "hi0", "lo1", "hi1"):
                        nodes[name] = nodes[name] + f32(0)
                    o["bottom-level nodes"] = nodes
                outs.append(o)
            _assert_equal(outs[1], outs[0], f"step {k}")
        assert outs[0]["hdr"].tobytes() != _frame_outputs_of_fresh(ggx_lut, s, w, h)["hdr"].tobytes(), "nothing moved"
    finally:
        for r in ctx:
            r.close()


def _frame_outputs_of_fresh(lut, s, w, h):
    with Renderer(w, h) as r:
        _upload_scene(r, lut, s)
        r.frame(s["camera"].frame_params(host.default_tonemap_params()))
        return {"hdr": r.read_hdr()}


# ---------------------------------------------------------------------------------------------------------- 2. lights
def test_lights_equal_host(ggx_lut):
    """Device-sourced light sets ((n * 48,) uint8 and (n, 12) float32 tensors, changing counts) against host-sourced ones:
    the cluster lists and the frames (shadow masks, G-buffer, HDR, sRGB8) byte for byte."""
    w, h = 480, 270
    s = scenes.shadow_scene(w, h)
    cam, tm = s["camera"], host.default_tonemap_params()
    versions = [_lights(s, k) for k in range(4)]
    dev = [_dev(v) if k % 2 else _dev(v.view(f32).reshape(len(v), 12)) for k, v in enumerate(versions)]
    _sync_torch()
    ctx = [Renderer(w, h), Renderer(w, h)]
    try:
        handles = []
        for r in ctx:
            _upload_scene(r, ggx_lut, s)
            handles.append(r.build_acceleration_structures())
        for k, v in enumerate(versions):
            ctx[0].set_lights(v)
            ctx[1].set_lights(dev[k])
            outs = []
            for r, hdl in zip(ctx, handles):
                r.frame(cam.frame_params(tm, acceleration_structure_address=hdl))
                o = _frame_outputs(r, True)
                o["cluster counts"], o["cluster indices"] = r.read_cluster_lights(_n_clusters(s))
                outs.append(o)
            _assert_equal(outs[1], outs[0], f"light set {k}")
            if k == 0:
                first = outs[0]["hdr"]
        assert first.tobytes() != outs[0]["hdr"].tobytes()
    finally:
        for r in ctx:
            r.close()


# ---------------------------------------------------------------------------------------------------------- 3. transforms
def test_transforms_equal_set_instances(ggx_lut):
    """8 animated frames on the config-4 scene (10 k instances, 64 lights, ray queries on): update_instance_transforms from
    device tensors (whole, partial, misaligned), pageable and page-locked arrays against set_instances of the full records,
    the top level updated on the host and on the device in turn: shadow masks, G-buffer, HDR and sRGB8 byte for byte."""
    import torch
    w, h = 480, 270
    s = scenes.instanced_scene(w, h)
    cam, tm = s["camera"], host.default_tonemap_params()
    n = len(s["instances"])
    ranges = [(0, n), (1000, 4000), (0, n), (n - 1, n), (2500, 9000), (0, n), (17, 18), (0, n)]
    sources = ["device", "device", "pageable", "device", "misaligned", "page-locked", "device", "device"]
    inst, frames, keep = s["instances"], [], []
    for f, ((a, b), kind) in enumerate(zip(ranges, sources)):
        inst = _rotated(inst, f, a, b)
        t = _transforms(inst[a:b])
        if kind == "device":
            src = _dev(t)
        elif kind == "misaligned":               # 4 bytes into a uint8 tensor: staged through the context's buffer
            buf = torch.zeros(t.nbytes + 16, dtype=torch.uint8, device="cuda")
            src = buf[4:4 + t.nbytes]
            src.copy_(torch.from_numpy(t.view(np.uint8).reshape(-1)).cuda())
            assert src.data_ptr() % 16 == 4
        elif kind == "page-locked":
            pin, src = _pinned(t)
            keep.append(pin)
        else:
            src = t
        frames.append((a, src, inst))
    _sync_torch()
    ctx = [Renderer(w, h), Renderer(w, h)]
    try:
        handles = []
        for r in ctx:
            _upload_scene(r, ggx_lut, s)
            handles.append(r.build_acceleration_structures())
        for f, (a, src, records) in enumerate(frames):
            ctx[0].set_instances(records)
            ctx[1].update_instance_transforms(src, first=a)
            outs = []
            for r, hdl in zip(ctx, handles):
                got = r.update_top_level_acceleration_structure_async() if f % 2 else r.update_top_level_acceleration_structure()
                assert got == hdl
                r.frame(cam.frame_params(tm, acceleration_structure_address=hdl))
                o = _frame_outputs(r, True)
                o["top-level records"] = _records_key(r.read_top_level_acceleration_structure()[1])
                outs.append(o)
            _assert_equal(outs[1], outs[0], f"frame {f} ({sources[f]} source, instances [{a}, {ranges[f][1]}))")
            if f == 0:
                first = outs[0]["layer 0 shadow mask"]
        assert (first != outs[0]["layer 0 shadow mask"]).any(0).mean() > 0.001, "the animation does not move the shadows"
        # ray queries off: the raster path alone
        for r in ctx:
            r.frame(cam.frame_params(tm))
        _assert_equal(_frame_outputs(ctx[1], False), _frame_outputs(ctx[0], False), "ray queries off")
    finally:
        for r in ctx:
            r.close()


# ---------------------------------------------------------------------------------------------------------- 4. stream order
@pytest.mark.parametrize("what", ["vertices", "lights", "transforms"])
def test_stream_order(ggx_lut, what):
    """The context stream is held up; frame A is enqueued, then a torch op on the context stream writes the new pose /
    lights / transforms into a device buffer, then the device-sourced update, then frame B: A shows the old state, B the
    new one."""
    import torch
    w, h = 480, 270
    s = scenes.shadow_scene(w, h)
    fp = s["camera"].frame_params(host.default_tonemap_params())
    if what == "vertices":
        new_pos, new_nrm, mesh = _deform(s["mesh"], 4, amp=0.1)
        s_new = dict(s, mesh=mesh)
        old_src, new_src = _dev(s["mesh"]["positions"]), _dev(new_pos)
        nrm = _dev(new_nrm)
        update = lambda r, d: r.update_mesh_vertices(d, nrm)
    elif what == "lights":
        s_new = dict(s, lights=_lights(s, 2))
        old_src, new_src = _dev(s["lights"]), _dev(s_new["lights"])
        update = lambda r, d: r.set_lights(d)
    else:
        s_new = dict(s, instances=_rotated(s["instances"], 6))
        old_src, new_src = _dev(_transforms(s["instances"])), _dev(_transforms(s_new["instances"]))
        update = lambda r, d: r.update_instance_transforms(d)
    want = []
    for sc in (s, s_new):
        with Renderer(w, h) as r:
            _upload_scene(r, ggx_lut, sc)
            r.frame(fp)
            want.append(r.read_srgb8())
    assert want[0].tobytes() != want[1].tobytes()
    stream = torch.cuda.Stream(device=0)
    d = old_src.clone()
    _sync_torch()
    a = torch.zeros(h * w * 4, dtype=torch.uint8).pin_memory().numpy().reshape(h, w, 4)
    with Renderer(w, h) as r:
        r.set_stream(stream.cuda_stream)
        _upload_scene(r, ggx_lut, s)
        r.frame(fp)
        r.sync()
        _hold(stream, 0.2)
        r.frame(fp)
        r.read_srgb8_async(a)
        with torch.cuda.stream(stream):
            d.copy_(new_src)                      # the producer, on the context stream behind the held-up frame
        update(r, d)
        r.frame(fp)
        r.wait_readback()
        b = r.read_srgb8()
        r.set_stream(None)
    assert a.tobytes() == want[0].tobytes(), "frame A saw the new state"
    assert b.tobytes() == want[1].tobytes(), "frame B did not see the state the stream produced"


# ---------------------------------------------------------------------------------------------------------- 5. same frame
def test_later_light_upload_wins(ggx_lut):
    """Two set_lights before one frame, one page-locked (run ahead on the upload stream) and one from device memory, in
    both orders: the frame shows the later one."""
    w, h = 480, 270
    s = scenes.instanced_scene(w, h, n_instances=3000, n_lights=32)
    fp = s["camera"].frame_params(host.default_tonemap_params())
    versions = [_lights(s, k) for k in range(3)]
    want = []
    for v in versions:
        with Renderer(w, h) as r:
            _upload_scene(r, ggx_lut, dict(s, lights=v))
            r.frame(fp)
            want.append(r.read_hdr())
    assert len({x.tobytes() for x in want}) == 3
    pins = [_pinned(v) for v in versions]
    dev = [_dev(v) for v in versions]
    _sync_torch()
    with Renderer(w, h) as r:
        _upload_scene(r, ggx_lut, s)
        r.frame(fp)
        r.set_lights(pins[1][1])                  # run ahead, then the device copy on the context stream
        r.set_lights(dev[2])
        r.frame(fp)
        r.sync()
        assert r.read_hdr().tobytes() == want[2].tobytes(), "page-locked then device: the device lights must win"
        r.set_lights(dev[0])                      # the device copy, then the run-ahead upload into the other buffer
        r.set_lights(pins[1][1])
        r.frame(fp)
        r.sync()
        assert r.read_hdr().tobytes() == want[1].tobytes(), "device then page-locked: the page-locked lights must win"
        for k in (2, 0, 1):                       # back to back, no sync: page-locked, then device, every frame
            r.set_lights(pins[(k + 1) % 3][1])
            r.set_lights(dev[k])
            r.frame(fp)
        r.sync()
        assert r.read_hdr().tobytes() == want[1].tobytes()


# ---------------------------------------------------------------------------------------------------------- 6. no blocking
def test_device_sources_do_not_block(ggx_lut):
    """With the stream held up on the GPU, device-sourced vertex, light and transform updates, the async top-level update
    and a traced frame return at once."""
    import torch
    w, h = 960, 540
    s = scenes.shadow_scene(w, h)
    fp = lambda hdl: s["camera"].frame_params(host.default_tonemap_params(), acceleration_structure_address=hdl)
    srcs = []
    for k in range(3):
        pos, nrm, _ = _deform(s["mesh"], k)
        srcs.append((_dev(pos), _dev(nrm), _dev(_lights(s, k)), _dev(_transforms(_rotated(s["instances"], k)))))
    _sync_torch()
    stream = torch.cuda.Stream(device=0)
    with Renderer(w, h) as r:
        r.set_stream(stream.cuda_stream)
        _upload_scene(r, ggx_lut, s)
        handle = r.build_acceleration_structures()

        def step(p, n, l, t):
            r.update_mesh_vertices(p, n)
            r.set_lights(l)
            r.update_instance_transforms(t)
            r.update_top_level_acceleration_structure_async()
            r.frame(fp(handle))

        for src in srcs[:2]:                      # warm-up: buffers at their sizes
            step(*src)
        r.sync()
        _hold(stream, 0.2)
        t0 = time.perf_counter()
        step(*srcs[2])
        enqueue = time.perf_counter() - t0
        r.sync()
        total = time.perf_counter() - t0
        r.set_stream(None)
    print(f"device sources: enqueue {enqueue * 1e3:.1f} ms, frame done after {total * 1e3:.1f} ms")
    assert total > 0.15, "the sleep did not hold up the stream"
    assert enqueue < 0.1, f"device-sourced updates + async top level + frame blocked for {enqueue * 1e3:.1f} ms"


# ---------------------------------------------------------------------------------------------------------- 7. group
def test_group_members_from_one_device_source(ggx_lut):
    """3 members on one device, each updated from the same device sources (vertices, lights, transforms) before
    tr_group_frame: the frame equals one context's, fed from host memory, bit for bit."""
    w, h = 960, 540
    s = scenes.shadow_scene(w, h)
    cam, tm = s["camera"], host.default_tonemap_params()
    pos, nrm, mesh = _deform(s["mesh"], 2, amp=0.1)
    lights, inst = _lights(s, 1), _rotated(s["instances"], 3)
    dpos, dnrm, dlights, dtr = _dev(pos), _dev(nrm), _dev(lights), _dev(_transforms(inst))
    _sync_torch()
    with Renderer(w, h) as r:
        _upload_scene(r, ggx_lut, dict(s, mesh=mesh, lights=lights, instances=inst))
        r.frame(cam.frame_params(tm, acceleration_structure_address=r.build_acceleration_structures()))
        want = r.read_hdr(), r.read_srgb8()
    members = [Renderer(w, h) for _ in range(3)]
    try:
        for m in members:
            _upload_scene(m, ggx_lut, s)
            m.build_acceleration_structures()
        with RendererGroup(members) as g:
            g.frame(cam.frame_params(tm, acceleration_structure_address=1))
            for m in members:
                m.update_mesh_vertices(dpos, dnrm)
                m.set_lights(dlights)
                m.update_instance_transforms(dtr)
                m.update_top_level_acceleration_structure_async()
            g.frame(cam.frame_params(tm, acceleration_structure_address=1))
            g.sync()
            got = g.read_hdr(), g.read_srgb8()
    finally:
        for m in members:
            m.close()
    assert got[0].tobytes() == want[0].tobytes(), "group HDR differs from one context"
    assert got[1].tobytes() == want[1].tobytes(), "group sRGB8 differs from one context"


# ---------------------------------------------------------------------------------------------------------- 8. rules
def test_rules(ggx_lut):
    import torch
    w, h = 160, 90
    s = scenes.shadow_scene(w, h)
    cam = s["camera"]
    n = len(s["instances"])
    t = _transforms(_rotated(s["instances"], 1))
    dt = _dev(t)
    _sync_torch()
    f = lib().tr_update_instance_transforms
    with Renderer(w, h) as r:
        with pytest.raises(TrError) as e:
            r.update_instance_transforms(t[:1])                      # no instances yet
        assert e.value.status == TR_ERR_INVALID_ARG
        _upload_scene(r, ggx_lut, s)
        handle = r.build_acceleration_structures()
        r.frame(cam.frame_params(acceleration_structure_address=handle))
        before_frame = r.read_hdr()
        for first, src in ((1, t), (n, t[:1]), (0, np.concatenate([t, t[:1]]))):
            with pytest.raises(TrError) as e:
                r.update_instance_transforms(src, first=first)
            assert e.value.status == TR_ERR_INVALID_ARG
        with pytest.raises(TrError) as e:
            r.update_instance_transforms(dt, first=1)
        assert e.value.status == TR_ERR_INVALID_ARG
        assert f(r._ctx, C.c_uint32(0), C.c_uint32(2), None) == TR_ERR_INVALID_ARG
        assert f(r._ctx, C.c_uint32(n), C.c_uint32(1), C.c_void_p(dt.data_ptr())) == TR_ERR_INVALID_ARG
        # the rejected calls changed nothing: the top level is still valid and the frame the same
        r.frame(cam.frame_params(acceleration_structure_address=handle))
        assert r.read_hdr().tobytes() == before_frame.tobytes()
        r.sync()
        before = Renderer.launch_count()
        assert f(r._ctx, C.c_uint32(n), C.c_uint32(0), None) == 0          # n = 0: nothing, even at the end
        r.update_instance_transforms(t[:0], first=3)
        assert Renderer.launch_count() == before
        r.update_instance_transforms(t)                                     # pageable: one launch
        assert Renderer.launch_count() - before == 1
        with pytest.raises(TrError) as e:                                   # traced frame without a top-level update
            r.frame(cam.frame_params(acceleration_structure_address=handle))
        assert e.value.status == TR_ERR_STATE
        r.frame(cam.frame_params())                                          # untraced frames still run
        before = Renderer.launch_count()
        r.update_instance_transforms(dt)                                    # device: one launch
        assert Renderer.launch_count() - before == 1
        assert r.update_top_level_acceleration_structure_async() == handle
        r.frame(cam.frame_params(acceleration_structure_address=handle))
        # non-finite values are accepted
        bad = t.copy()
        bad[0, 0], bad[1, 4] = np.nan, np.inf
        r.update_instance_transforms(_dev(bad))
        r.sync()
        # what renderer.py refuses before the call: wrong dtype, shape or layout
        with pytest.raises(TypeError):
            r.update_instance_transforms(dt.double())
        with pytest.raises(ValueError):
            r.update_instance_transforms(dt[:, :4])
        with pytest.raises(ValueError):
            r.update_instance_transforms(dt.t().contiguous().t())
        with pytest.raises(ValueError):
            r.set_lights(_dev(s["lights"])[:47])
        with pytest.raises(TypeError):
            r.update_mesh_vertices(torch.zeros((4, 3), dtype=torch.float64, device="cuda"), torch.zeros((4, 3), device="cuda"))
        with pytest.raises(ValueError):
            r.update_mesh_vertices(torch.zeros((4, 3), device="cuda"), torch.zeros((5, 3), device="cuda"))
        # a null device array of zero rows is n = 0
        r.update_mesh_vertices(torch.zeros((0, 3), device="cuda"), torch.zeros((0, 3), device="cuda"))
    if torch.cuda.device_count() < 2:
        return
    with Renderer(w, h, device=0) as r:
        _upload_scene(r, ggx_lut, s)
        with pytest.raises(ValueError):
            r.update_instance_transforms(dt.to("cuda:1"))
        with pytest.raises(ValueError):
            r.set_lights(_dev(s["lights"]).to("cuda:1"))
