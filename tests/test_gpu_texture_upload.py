"""tr_set_texture_async: a material image bound from its level 0, the mip chain built on the device in stream order
(csrc/k_textures.cu), against the blocking tr_set_texture fed the Python ingest's CPU chain (scenes.make_mips).

The store the samplers read must be bit-equal level by level, and so must every frame that samples it.  The call is
stream-ordered (the frame before it samples the old image, the next one the new), never waits with a page-locked source
unless a bound index has to grow, and launches one kernel per level."""
import ctypes as C
import time

import numpy as np
import pytest

from accel_checks import _hold, _pinned, _upload_scene
from transmission_renderer_b200 import Renderer, RendererGroup, TrError, host, scenes
from transmission_renderer_b200.renderer import _lib
from test_texture_chain_rule import SIZES, image

pytestmark = pytest.mark.gpu

TR_ERR_INVALID_ARG, TR_ERR_STATE = -1, -6


def _bind_blocking(r, index, img, srgb, n_levels=0):
    levels = scenes.make_mips(img, srgb)
    r.set_texture(index, levels[: n_levels or len(levels)], srgb)


def _levels(r, index):
    out, k = [], 0
    while True:
        try:
            out.append(r.read_texture_level(index, k))
        except TrError as e:
            assert e.status == TR_ERR_INVALID_ARG
            return out
        k += 1


# ------------------------------------------------------------------------------------------------ 1. the store
@pytest.mark.parametrize("size", SIZES, ids=[f"{w}x{h}" for w, h in SIZES])
def test_store_equals_blocking_make_mips(size):
    """Every level of the store, sRGB and UNORM, n_levels 0 (full), 1 and full - 1; pinned and pageable sources."""
    w, h = size
    full = host.mip_levels_for_size(w, h)
    with Renderer(64, 64) as r:
        for srgb in (True, False):
            for kind in ("random", "gradient"):
                img = image(kind, w, h, seed=11 if srgb else 12)
                chain = scenes.make_mips(img, srgb)
                keep, pin = _pinned(img)
                for n in sorted({0, 1, max(full - 1, 1)}):
                    r.set_texture_async(0, pin if kind == "random" else img, srgb, n_levels=n)
                    r.set_texture(1, chain[: n or full], srgb)
                    got, want = _levels(r, 0), _levels(r, 1)
                    assert len(got) == len(want) == (n or full)
                    for k, (g, x) in enumerate(zip(got, want)):
                        assert g.shape == x.shape
                        assert g.tobytes() == x.tobytes(), \
                            f"{w}x{h} srgb={srgb} {kind} n_levels={n} level {k}: {(g != x).any(-1).sum()} texels differ"
                del keep


# ------------------------------------------------------------------------------------------------ 2. frames
def _gltf_scene(tmp_path, w, h):
    from test_gltf_ingest import _asset
    from transmission_renderer_b200 import gltf_ingest
    path, _ = _asset(tmp_path)
    s = gltf_ingest.finish(gltf_ingest.load_gltf(path))
    s.update(camera=scenes.Camera(w, h, (0.0, 3.0, 6.0), 0.0, -15.0), lights=scenes.config2_lights(),
             uniforms=host.make_uniforms(w, h))
    return s


def _render(s, lut, on_device, traced, f32=True):
    w, h = s["camera"].width, s["camera"].height
    with Renderer(w, h, f32_debug=f32) as r:
        keep = [_pinned(t["levels"][0]) for t in s["textures"]] if on_device else []
        if on_device:
            for i, (t, (_, pin)) in enumerate(zip(s["textures"], keep)):
                r.set_texture_async(i, pin, t["srgb"])
        else:
            r.set_textures(s["textures"])
        _upload_scene(r, lut, s)
        handle = r.build_acceleration_structures() if traced else 0
        r.frame(s["camera"].frame_params(host.default_tonemap_params(), acceleration_structure_address=handle))
        out = {f"g{layer}_{k}": v for layer in (0, 1) for k, v in r.read_gbuffer(layer, derivatives=True).items()
               if v is not None}
        out.update(hdr=r.read_hdr(), srgb8=r.read_srgb8())
        if f32:
            out["hdr_f32"] = r.read_hdr_f32()
        r.sync()
    return out


@pytest.mark.parametrize("traced", [False, True], ids=["raster", "ray_queries"])
@pytest.mark.parametrize("scene", ["textured_spheres", "alpha_clip", "gltf"])
def test_frames_equal_blocking_binding(ggx_lut, tmp_path, scene, traced):
    """Level 0 only, bound on the device: G-buffer planes (duv included), fp16 and fp32 HDR and sRGB8 byte-equal to the
    frame of the blocking binding of make_mips's chains."""
    w, h = 480, 270
    s = {"textured_spheres": lambda: scenes.textured_sphere_scene(w, h), "alpha_clip": lambda: scenes.alpha_clip_scene(w, h),
         "gltf": lambda: _gltf_scene(tmp_path, w, h)}[scene]()
    want = _render(s, ggx_lut, on_device=False, traced=traced)
    got = _render(s, ggx_lut, on_device=True, traced=traced)
    assert set(got) == set(want) and "g0_duv" in got
    for k in want:
        assert got[k].tobytes() == want[k].tobytes(), f"{k}: {(got[k] != want[k]).sum()} values differ"
    assert np.abs(want["g0_duv"]).max() > 1e-3   # the level of detail is exercised


# ------------------------------------------------------------------------------------------------ 3. ordering
def _other_image(w, h, seed):
    return image("random", w, h, seed=seed)


def _textured_frame(s, lut, bind):
    """sRGB8 of one frame of `s` with the diffuse image (index 0) bound by `bind(r)` after the others (blocking)."""
    w, h = s["camera"].width, s["camera"].height
    with Renderer(w, h) as r:
        r.set_textures(s["textures"])
        bind(r)
        _upload_scene(r, lut, s)
        r.frame(s["camera"].frame_params(host.default_tonemap_params()))
        return r.read_srgb8()


@pytest.mark.parametrize("case", ["same_size", "grow", "shrink", "blocking_then_async", "async_then_blocking"])
def test_frame_before_sees_old_image_frame_after_new(ggx_lut, case):
    """Frame A, read_srgb8_async, a rebind of the diffuse image A samples, frame B: A shows the old image, B the new,
    with the stream held up so that A is still queued when the rebind is enqueued."""
    import torch
    w, h = 320, 180
    s = scenes.textured_sphere_scene(w, h)
    side = {"same_size": (256, 256), "grow": (512, 512), "shrink": (128, 64)}.get(case, (256, 256))
    old = s["textures"][0]["levels"][0]
    new = _other_image(*side, seed=41)
    want_a = _textured_frame(s, ggx_lut, lambda r: None)
    want_b = _textured_frame(s, ggx_lut, lambda r: _bind_blocking(r, 0, new, True))
    assert (want_a != want_b).any()
    keep_old, pin_old = _pinned(old)
    keep_new, pin_new = _pinned(new)
    stream = torch.cuda.Stream(device=0)
    with Renderer(w, h) as r:
        r.set_stream(stream.cuda_stream)
        r.set_textures(s["textures"])
        if case != "blocking_then_async":       # the rebinds below then fit (same size, shrink) or grow an async binding
            r.set_texture_async(0, pin_old, True)
        _upload_scene(r, ggx_lut, s)
        fp = s["camera"].frame_params(host.default_tonemap_params())
        r.frame(fp)                              # warm-up: frame buffers
        r.sync()
        keep_a, out_a = _pinned(np.zeros((h, w, 4), np.uint8))
        _hold(stream, 0.05)
        r.frame(fp)                              # A
        r.read_srgb8_async(out_a)
        if case == "async_then_blocking":
            _bind_blocking(r, 0, new, True)
        else:
            r.set_texture_async(0, pin_new, True)
        r.frame(fp)                              # B
        got_b = r.read_srgb8()
        r.wait_readback()
        r.set_stream(None)
    assert out_a.tobytes() == want_a.tobytes(), f"{case}: frame A does not show the old image"
    assert got_b.tobytes() == want_b.tobytes(), f"{case}: frame B does not show the new image"
    del keep_old, keep_new, keep_a


# ------------------------------------------------------------------------------------------------ 4. no wait
def test_first_binds_do_not_wait_growing_rebind_does(ggx_lut):
    """With the stream held for 0.2 s: 16 first-time binds of page-locked 512x512 images plus a frame enqueue return at
    once; a rebind that needs a larger allocation waits for the stream."""
    import torch
    w, h = 640, 360
    s = scenes.textured_sphere_scene(w, h)
    imgs = [_pinned(image("random", 512, 512, seed=100 + i)) for i in range(16)]
    big = _pinned(image("random", 1024, 1024, seed=99))
    stream = torch.cuda.Stream(device=0)
    with Renderer(w, h) as r:
        r.set_stream(stream.cuda_stream)
        for i, t in enumerate(s["textures"]):
            r.set_texture_async(i, t["levels"][0], t["srgb"])
        _upload_scene(r, ggx_lut, s)
        fp = s["camera"].frame_params(host.default_tonemap_params())
        r.frame(fp)
        r.sync()
        _hold(stream, 0.2)
        t0 = time.perf_counter()
        for i, (_, pin) in enumerate(imgs):
            r.set_texture_async(8 + i, pin, i % 2 == 0)
        binds = time.perf_counter() - t0
        r.frame(fp)
        enqueue = time.perf_counter() - t0
        r.sync()
        total = time.perf_counter() - t0
        _hold(stream, 0.2)
        t0 = time.perf_counter()
        r.set_texture_async(8, big[1], True)
        grow = time.perf_counter() - t0
        r.sync()
        got = r.read_texture_level(8, 3)
        _bind_blocking(r, 9, big[1], True)
        assert got.tobytes() == r.read_texture_level(9, 3).tobytes()
        r.set_stream(None)
    print(f"16 first binds {binds * 1e3:.1f} ms, + frame: enqueue {enqueue * 1e3:.1f} ms, done after {total * 1e3:.1f} ms; growing rebind "
          f"{grow * 1e3:.1f} ms")
    assert total > 0.15, "the sleep did not hold up the stream"
    assert enqueue < 0.1, f"first-time binds + frame blocked for {enqueue * 1e3:.1f} ms"
    assert grow > 0.15, "a rebind that grows the allocation must wait for the frame in flight"


# ------------------------------------------------------------------------------------------------ 5. launches
def test_one_launch_per_level():
    img = image("random", 300, 200)
    full = host.mip_levels_for_size(300, 200)
    with Renderer(64, 64) as r:
        for n in (0, 1, 3, full):
            before = Renderer.launch_count()
            r.set_texture_async(2, img, n % 2 == 0, n_levels=n)
            assert Renderer.launch_count() - before == (n or full)
        before = Renderer.launch_count()
        _bind_blocking(r, 3, img, True)
        assert Renderer.launch_count() == before


# ------------------------------------------------------------------------------------------------ 6. errors
def test_rejected_arguments_change_nothing():
    img = image("random", 64, 64)
    with Renderer(64, 64) as r:
        r.set_texture_async(0, img, True)
        want = _levels(r, 0)
        lib, ctx = _lib(), r._ctx
        p = img.ctypes.data_as(C.c_void_p)
        cases = [  # (index, pointer, w, h, n_levels)
            (193, p, 64, 64, 0), (0, None, 64, 64, 0), (0, p, 0, 64, 0), (0, p, 64, 0, 0), (0, p, 64, 64, 17),
            (0, p, 64, 64, 8),   # the full chain of 64x64 is 7 levels
        ]
        for idx, ptr, w, h, n in cases:
            before = Renderer.launch_count()
            st = lib.tr_set_texture_async(ctx, C.c_uint32(idx), ptr, C.c_uint32(w), C.c_uint32(h), C.c_int32(0), C.c_uint32(n))
            assert st == TR_ERR_INVALID_ARG, (idx, w, h, n, st)
            assert Renderer.launch_count() == before
        r.set_texture_async(1, image("random", 16, 16), False, n_levels=5)   # 16x16: full chain, accepted
        got = _levels(r, 0)
        assert [g.tobytes() for g in got] == [x.tobytes() for x in want]
        with pytest.raises(TrError) as e:
            r.read_texture_level(5, 0)
        assert e.value.status == TR_ERR_STATE
        with pytest.raises(TrError) as e:
            r.read_texture_level(193, 0)
        assert e.value.status == TR_ERR_INVALID_ARG
        with pytest.raises(TrError) as e:
            r.read_texture_level(0, 7)
        assert e.value.status == TR_ERR_INVALID_ARG


# ------------------------------------------------------------------------------------------------ 7. group
def test_group_members_bind_on_device(ggx_lut):
    """A 3-member tr_group whose members bind level 0 only renders the frame of one context with the blocking binding."""
    w, h = 480, 270
    s = scenes.textured_sphere_scene(w, h)
    fp = s["camera"].frame_params(host.default_tonemap_params())
    with Renderer(w, h) as r:
        r.set_textures(s["textures"])
        _upload_scene(r, ggx_lut, s)
        r.frame(fp)
        want = r.read_hdr(), r.read_srgb8()
    keep = [_pinned(t["levels"][0]) for t in s["textures"]]
    members = [Renderer(w, h) for _ in range(3)]
    try:
        for r in members:
            for i, (t, (_, pin)) in enumerate(zip(s["textures"], keep)):
                r.set_texture_async(i, pin, t["srgb"])
            _upload_scene(r, ggx_lut, s)
        with RendererGroup(members) as g:
            g.frame(fp)
            got = g.read_hdr(), g.read_srgb8()
    finally:
        for r in members:
            r.close()
    assert got[0].tobytes() == want[0].tobytes(), "group HDR differs from the blocking binding"
    assert got[1].tobytes() == want[1].tobytes(), "group sRGB8 differs from the blocking binding"
