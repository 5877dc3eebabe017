"""Single-process groups (tr_group_*): n contexts of one host thread render the bands of one frame, each storing its opaque band
into every member's mip 0, ordered by CUDA events.  On one device the members run exactly the code n GPUs run, so the fused
peer-store exchange is checked here bit for bit against one context rendering the whole frame."""
import ctypes as C
import time

import numpy as np
import pytest

from pipeline import gpu_setup
from transmission_renderer_b200 import Renderer, RendererGroup, TrError, abi, host, lib, scenes

pytestmark = pytest.mark.gpu

W, H = 1920, 1080
YAWS = (0.0, 7.5, 15.0)
TR_ERR_INVALID_ARG, TR_ERR_STATE = -1, -6


def _upload(r, lut, s):
    gpu_setup(r, lut, s["uniforms"], s["materials"], s["lights"])
    r.set_instances(s["instances"])
    r.set_primitives(s["primitives"])
    m = s["mesh"]
    r.set_mesh(m["positions"], m["normals"], m["uvs"], m["indices"])
    r.build_clusters(s["camera"].write_cluster_data())


def _params(w, h, yaw):
    # the camera of scenes.instanced_scene, turned by `yaw`
    return scenes.Camera(w, h, (0.0, 6.0, 0.0), yaw, -10.0).frame_params(host.default_tonemap_params())


def _single(lut, s, w, h, frames):
    """One context, whole frame: (hdr, srgb, mip0) after each of `frames`."""
    out = []
    with Renderer(w, h) as r:
        _upload(r, lut, s)
        for fp in frames:
            r.frame(fp)
            out.append((r.read_hdr(), r.read_srgb8(), r.read_pyramid_level(0)))
    return out


def _assert_same(g, ref, label):
    hdr, srgb, mip0 = ref
    got = g.read_hdr()
    assert got.tobytes() == hdr.tobytes(), f"{label}: HDR differs in {(got != hdr).any(axis=2).sum()} pixels"
    assert g.read_srgb8().tobytes() == srgb.tobytes(), f"{label}: sRGB8 differs"
    for k, r in enumerate(g.renderers):
        assert r.read_pyramid_level(0).tobytes() == mip0.tobytes(), f"{label}: member {k}'s mip 0 differs"


@pytest.fixture(scope="module")
def scene():
    return scenes.instanced_scene(W, H)


@pytest.fixture(scope="module")
def single_frames(ggx_lut, scene):
    return _single(ggx_lut, scene, W, H, [_params(W, H, y) for y in YAWS])


@pytest.mark.parametrize("n", [2, 3, 8])
def test_group_on_one_device_equals_one_context(ggx_lut, scene, single_frames, n):
    """n members on device 0 (ragged bands for n = 3): every frame's stitched HDR, group sRGB8 and every member's mip 0 are
    the single context's bytes; then the three frames again back to back, so a frame's opaque stores overlap the previous
    frame's transmissive pass of the other members, and the last one must still be the same."""
    members = [Renderer(W, H) for _ in range(n)]
    try:
        for r in members:
            _upload(r, ggx_lut, scene)
        with RendererGroup(members) as g:
            if n == 3:
                g.set_bands([0, 8, 600, H])
            for yaw, ref in zip(YAWS, single_frames):
                g.frame(_params(W, H, yaw))
                _assert_same(g, ref, f"n={n} yaw {yaw}")
            for yaw in YAWS:
                g.frame(_params(W, H, yaw))
            g.sync()
            _assert_same(g, single_frames[-1], f"n={n} back to back")
    finally:
        for r in members:
            r.close()


def test_group_resize_then_frame(ggx_lut, scene):
    w, h = 1280, 720
    s720 = scenes.instanced_scene(w, h)
    ref = _single(ggx_lut, s720, w, h, [_params(w, h, 0.0)])[0]
    members = [Renderer(W, H) for _ in range(3)]
    try:
        for r in members:
            _upload(r, ggx_lut, scene)
        with RendererGroup(members) as g:
            g.frame(_params(W, H, 0.0))
            g.resize(w, h)
            assert g.bounds == [0, 240, 480, 720]
            for r in members:   # the reference re-runs write_cluster_data with the new cluster size on resize (main.rs:1113-1121)
                r.set_uniforms(s720["uniforms"])
                r.build_clusters(s720["camera"].write_cluster_data())
            g.frame(_params(w, h, 0.0))
            _assert_same(g, ref, "after tr_group_resize")
    finally:
        for r in members:
            r.close()


def test_group_ray_queried_shadows(ggx_lut):
    w, h = 960, 540
    s = scenes.shadow_scene(w, h)
    cam = s["camera"]
    with Renderer(w, h) as r:
        _upload(r, ggx_lut, s)
        r.frame(cam.frame_params(host.default_tonemap_params(), acceleration_structure_address=r.build_acceleration_structures()))
        ref = (r.read_hdr(), r.read_srgb8(), r.read_pyramid_level(0))
        masks = [r.read_shadow_mask(0), r.read_shadow_mask(1)]
    members = [Renderer(w, h) for _ in range(3)]
    try:
        for r in members:
            _upload(r, ggx_lut, s)
            r.build_acceleration_structures()
        with RendererGroup(members) as g:
            assert len({r.acceleration_structure_address for r in members}) == 3
            per_member = [cam.frame_params(host.default_tonemap_params(), acceleration_structure_address=r.acceleration_structure_address)
                          for r in members]
            g.frame(per_member)
            _assert_same(g, ref, "ray queries, per-member params")
            for k, r in enumerate(members):
                y0, y1 = g.bounds[k], g.bounds[k + 1]
                for layer in (0, 1):
                    assert r.read_shadow_mask(layer)[:, y0:y1].tobytes() == masks[layer][:, y0:y1].tobytes(), \
                        f"member {k} layer {layer}: shadow bits differ"
            # one struct for all: the group puts in each member's own handle
            g.frame(cam.frame_params(host.default_tonemap_params(), acceleration_structure_address=members[0].acceleration_structure_address))
            _assert_same(g, ref, "ray queries, broadcast params")
    finally:
        for r in members:
            r.close()


def test_group_adds_no_kernels(ggx_lut, scene):
    """A group frame launches exactly the kernels its members launch rendering their bands alone: no barrier kernel, no
    copy kernel; the exchange is the opaque pass's own stores."""
    n = 3
    fp = _params(W, H, 0.0)
    alone = 0
    for k in range(n):
        with Renderer(W, H) as r:
            _upload(r, ggx_lut, scene)
            r.set_band(*host.band_rows(H, k, n))
            r.frame(fp)
            r.frame(fp)
            r.sync()
            before = Renderer.launch_count()
            r.frame(fp)
            r.sync()
            alone += Renderer.launch_count() - before
    members = [Renderer(W, H) for _ in range(n)]
    try:
        for r in members:
            _upload(r, ggx_lut, scene)
        with RendererGroup(members) as g:
            g.frame(fp)
            g.frame(fp)
            g.sync()
            before = Renderer.launch_count()
            g.frame(fp)
            g.sync()
            grouped = Renderer.launch_count() - before
    finally:
        for r in members:
            r.close()
    assert grouped == alone, f"group frame launched {grouped} kernels, its members alone {alone}"


def test_group_frame_does_not_block(ggx_lut, scene):
    """With member 0's stream held up on the GPU, tr_group_frame still returns at once: every ordering is a GPU-side event
    wait, nothing on the host waits for the device."""
    import torch
    stream = torch.cuda.Stream(device=0)
    members = [Renderer(W, H) for _ in range(2)]
    try:
        for r in members:
            _upload(r, ggx_lut, scene)
        members[0].set_stream(stream.cuda_stream)
        fp = _params(W, H, 0.0)
        with RendererGroup(members) as g:
            for _ in range(2):
                g.frame(fp)
            g.sync()
            clock_khz = getattr(torch.cuda.get_device_properties(0), "clock_rate", 0) or 2_100_000
            with torch.cuda.stream(stream):
                torch.cuda._sleep(int(0.2 * clock_khz * 1e3))   # >= 0.2 s: the cycles at the highest clock
            t0 = time.perf_counter()
            g.frame(fp)
            enqueue = time.perf_counter() - t0
            g.sync()
            total = time.perf_counter() - t0
        members[0].set_stream(None)
    finally:
        for r in members:
            r.close()
    print(f"tr_group_frame returned after {enqueue * 1e3:.1f} ms; the frame finished after {total * 1e3:.1f} ms")
    assert total > 0.15, "the sleep did not hold up member 0's stream"
    assert enqueue < 0.1, f"tr_group_frame blocked for {enqueue * 1e3:.1f} ms"


def _status(fn, *args):
    st = fn(*args)
    return st, lib().tr_last_error().decode()


def test_group_rules(ggx_lut):
    w, h = 320, 180
    s = scenes.instanced_scene(w, h, n_instances=2000, n_lights=16)
    fp = s["camera"].frame_params(host.default_tonemap_params())
    a, b, c = (Renderer(w, h) for _ in range(3))
    odd = Renderer(w, h + 8)
    many = [Renderer(64, 32) for _ in range(9)]
    groups = []
    try:
        for bad, status in (([a, a], TR_ERR_INVALID_ARG), ([a, odd], TR_ERR_INVALID_ARG), ([], TR_ERR_INVALID_ARG),
                            (many, TR_ERR_INVALID_ARG)):
            with pytest.raises(TrError) as e:
                RendererGroup(bad)
            assert e.value.status == status, str(e.value)
        for r in (a, b, c):
            _upload(r, ggx_lut, s)
        g = RendererGroup([a, b])
        groups.append(g)
        with pytest.raises(TrError) as e:
            RendererGroup([b, c])
        assert e.value.status == TR_ERR_STATE and "another group" in str(e.value)

        L = lib()
        ctx = b._ctx
        pc = np.ascontiguousarray(fp["push_constants"])
        bounds = np.array([0, h], np.uint32)
        uid = (C.c_uint8 * 128)()
        handles = (C.c_uint8 * 128)()
        calls = {
            "tr_frame": (L.tr_frame, ctx, fp.ctypes.data_as(C.c_void_p)),
            "tr_shade_opaque": (L.tr_shade_opaque, ctx, pc.ctypes.data_as(C.c_void_p)),
            "tr_allgather_opaque": (L.tr_allgather_opaque, ctx),
            "tr_set_band": (L.tr_set_band, ctx, C.c_uint32(0), C.c_uint32(h)),
            "tr_set_bands": (L.tr_set_bands, ctx, bounds.ctypes.data_as(C.c_void_p), C.c_uint32(2)),
            "tr_resize": (L.tr_resize, ctx, C.c_uint32(w), C.c_uint32(h)),
            "tr_comm_init": (L.tr_comm_init, ctx, uid, C.c_int32(0), C.c_int32(2)),
            "tr_peer_attach": (L.tr_peer_attach, ctx, C.c_int32(1), C.c_int32(2), handles),
            "tr_destroy": (L.tr_destroy, ctx),
        }
        for name, (fn, *args) in calls.items():
            st, msg = _status(fn, *args)
            assert st == TR_ERR_STATE and "tr_group" in msg, (name, st, msg)
        # still a working member after the refused tr_destroy
        g.frame(fp)
        g.sync()
        group_srgb = g.read_srgb8()
        g.close()

        with Renderer(w, h) as fresh:
            _upload(fresh, ggx_lut, s)
            fresh.frame(fp)
            want = (fresh.read_hdr(), fresh.read_srgb8(), fresh.read_pyramid_level(0))
        assert group_srgb.tobytes() == want[1].tobytes()
        for k, r in enumerate((a, b)):   # whole-frame contexts again
            r.frame(fp)
            got = (r.read_hdr(), r.read_srgb8(), r.read_pyramid_level(0))
            assert all(x.tobytes() == y.tobytes() for x, y in zip(got, want)), f"former member {k} differs from a fresh context"
    finally:
        for g in groups:
            g.close()
        for r in (a, b, c, odd, *many):
            r.close()


def test_group_across_devices(ggx_lut, scene, single_frames):
    import torch
    n_dev = torch.cuda.device_count()
    if n_dev < 2:
        pytest.skip("needs at least 2 GPUs")
    for devices in (list(range(min(8, n_dev))), [d for d in range(min(4, n_dev)) for _ in range(2)]):
        members = [Renderer(W, H, device=d) for d in devices]
        try:
            for r in members:
                _upload(r, ggx_lut, scene)
            with RendererGroup(members) as g:
                for yaw, ref in zip(YAWS, single_frames):
                    g.frame(_params(W, H, yaw))
                    _assert_same(g, ref, f"devices {devices} yaw {yaw}")
        finally:
            for r in members:
                r.close()
