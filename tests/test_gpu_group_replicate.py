"""tr_group_replicate_scene: one member of a group is loaded, and the library copies its scene into every other member, GPU
to GPU in stream order.  The reference for every comparison is a group whose members were each loaded directly with the
same arrays and built the same structures; every comparison is byte equality."""
import ctypes as C
import time

import numpy as np
import pytest

from accel_checks import _deform, _hold, _pinned, _upload_scene
from transmission_renderer_b200 import Renderer, RendererGroup, TrError, host, scenes
from transmission_renderer_b200.renderer import _lib

pytestmark = pytest.mark.gpu

W, H = 480, 270
TR_ERR_INVALID_ARG, TR_ERR_STATE = -1, -6
RT = ["none", "host", "async", "refit"]


# ---------------------------------------------------------------------------------------------------------- scenes
def _config4_textured(w, h):
    """Config 4 (2 000 instances, 64 lights) with texture-mapped materials, and the box and glass-sphere primitives drawn
    with the alpha test (draw buffers 1 and 3)."""
    s = scenes.instanced_scene(w, h, n_instances=2000)
    s["textures"] = scenes.procedural_textures(128)
    mats = s["materials"]
    for m in range(len(mats)):
        if m % 3 == 0:
            mats["textures"][m, scenes.TEX_SLOTS["diffuse"]] = 0
            mats["alpha_clipping_cutoff"][m] = 0.5
        if m % 4 == 1:
            mats["textures"][m, scenes.TEX_SLOTS["normal_map"]] = 2
            mats["textures"][m, scenes.TEX_SLOTS["metallic_roughness"]] = 1
        if m % 5 == 2:
            mats["textures"][m, scenes.TEX_SLOTS["emissive"]] = 3
            mats["emissive_factor"][m, :3] = (1.5, 1.5, 1.5)
    prims = s["primitives"]
    prims["draw_buffer_index"][1] = 1
    prims["draw_buffer_index"][6] = 3
    s["pitch"] = -10.0
    return s


def _gltf(tmp_path, w, h):
    from test_gpu_texture_upload import _gltf_scene
    s = _gltf_scene(tmp_path, w, h)
    s["pitch"] = -15.0
    return s


SCENES = {"config4": lambda tmp, w, h: _config4_textured(w, h), "gltf": lambda tmp, w, h: _gltf(tmp, w, h)}


# ---------------------------------------------------------------------------------------------------------- loading
def _bind_textures(r, s, keep):
    """Even images bound by tr_set_texture_async from page-locked level 0 (the store holds their RGBA8 levels too), odd
    ones by the blocking tr_set_texture."""
    for i, t in enumerate(s.get("textures", [])):
        if i % 2 == 0:
            if i not in keep:
                keep[i] = _pinned(t["levels"][0])
            r.set_texture_async(i, keep[i][1], t["srgb"])
        else:
            r.set_texture(i, t["levels"], t["srgb"])


def _load(r, lut, s, rt, keep):
    """Everything a frame needs, the way the reference loads a context, then the structures of variant `rt`."""
    _bind_textures(r, s, keep)
    _upload_scene(r, lut, s)
    if rt == "host":
        r.build_acceleration_structures()
    elif rt in ("async", "refit"):
        r.build_acceleration_structures_async()
    if rt == "refit":
        p, n, _ = _deform(s["mesh"], 1)
        r.update_mesh_vertices(p, n)   # refits the trees; the top level waits for its update


def _finish(members, rt):
    """After the load (direct or replicated): the refit variant's top-level update on every member."""
    if rt == "refit":
        for r in members:
            r.update_top_level_acceleration_structure_async()


def _params(s, members, rt, yaw=0.0):
    """One frame-params struct per member, with the member's own handle when ray queries are on; `yaw` turns the camera."""
    cam = s["camera"]
    if yaw:
        cam = scenes.Camera(cam.width, cam.height, cam.position, yaw, s["pitch"])
    return [cam.frame_params(host.default_tonemap_params(), acceleration_structure_address=r.acceleration_structure_address if rt != "none" else 0)
            for r in members]


def _capture(g, textured):
    out = dict(hdr=g.read_hdr(), srgb8=g.read_srgb8())
    for k, r in enumerate(g.renderers):
        for layer in (0, 1):
            for name, v in r.read_gbuffer(layer, derivatives=textured).items():
                if v is not None:
                    out[f"m{k}_g{layer}_{name}"] = v
    return out


def _masks(g):
    return {f"m{k}_mask{layer}": r.read_shadow_mask(layer) for k, r in enumerate(g.renderers) for layer in (0, 1)}


def _assert_equal(got, want, label):
    assert set(got) == set(want), label
    for k in want:
        assert got[k].tobytes() == want[k].tobytes(), f"{label}: {k} differs in {(got[k] != want[k]).sum()} values"


def _state(r, s, rt):
    """What a member holds of the scene, as its parity hooks read it."""
    out = {"spheres": r.read_chunk_spheres()}
    for i, t in enumerate(s.get("textures", [])):
        for k in range(len(t["levels"])):
            out[f"tex{i}_{k}"] = r.read_texture_level(i, k)
    if rt != "none":
        out["blas_nodes"], out["blas_tris"] = r.read_bottom_level_acceleration_structure()
        out["tlas_nodes"], out["tlas_inst"] = r.read_top_level_acceleration_structure()
    return out


class _Groups:
    """A directly loaded group and a replicated one over the same scene, on `devices`."""

    def __init__(self, lut, s, rt, devices, source):
        self.keep = {}
        self.direct = [Renderer(W, H, device=d) for d in devices]
        self.rep = [Renderer(W, H, device=d) for d in devices]
        self.groups = []
        for r in self.direct:
            _load(r, lut, s, rt, self.keep)
        self.gd = RendererGroup(self.direct)
        self.groups.append(self.gd)
        self.gr = RendererGroup(self.rep)
        self.groups.append(self.gr)
        _load(self.rep[source], lut, s, rt, self.keep)
        self.addresses = self.gr.replicate_scene(source)
        _finish(self.direct, rt)
        _finish(self.rep, rt)

    def close(self):
        for g in self.groups:
            g.close()
        for r in self.direct + self.rep:
            r.close()


# ---------------------------------------------------------------------------------------------------------- 1 + 2
@pytest.mark.parametrize("rt", RT)
@pytest.mark.parametrize("scene", ["config4", "gltf"])
def test_same_frames_and_state(ggx_lut, tmp_path, scene, rt):
    """Two yaws of group frames: stitched HDR and sRGB8, every member's G-buffer planes and, with ray queries, its shadow
    masks; then every destination's images (every level), culling spheres and both tree levels against the source's."""
    s = SCENES[scene](tmp_path, W, H)
    n, source = (3, 1) if rt in ("none", "async") else (2, 0)
    gs = _Groups(ggx_lut, s, rt, [0] * n, source)
    try:
        if rt in ("none", "refit"):   # refit: the source's top level waits for its update, which each member makes itself
            assert gs.addresses == [0] * n
        else:
            assert all(gs.addresses) and len(set(gs.addresses)) == n
        for yaw in (0.0, 9.0):
            gs.gd.frame(_params(s, gs.direct, rt, yaw))
            gs.gr.frame(_params(s, gs.rep, rt, yaw))
            want, got = _capture(gs.gd, "textures" in s), _capture(gs.gr, "textures" in s)
            if rt != "none":
                want.update(_masks(gs.gd))
                got.update(_masks(gs.gr))
            _assert_equal(got, want, f"{scene} {rt} yaw {yaw}")
        ref = _state(gs.rep[source], s, rt)
        for k, r in enumerate(gs.rep):
            if k != source:
                _assert_equal(_state(r, s, rt), ref, f"{scene} {rt}: member {k}'s state")
        _assert_equal(_state(gs.direct[source], s, rt), ref, f"{scene} {rt}: the directly loaded member")
    finally:
        gs.close()


# ---------------------------------------------------------------------------------------------------------- 3
def _animate(members, s, k):
    """Frame k of the animation on every member: a quarter of the instances turned and moved, the mesh displaced, then
    the async top-level update."""
    inst = s["instances"]
    first, n = 100, len(inst) // 4
    t = np.zeros((n, 8), np.float32)
    t[:, :4] = inst["translation_and_scale"][first:first + n]
    t[:, 0] += np.float32(0.3 * np.sin(0.5 * k))
    angle = 0.2 * k
    t[:, 4:] = (0.0, np.sin(angle / 2), 0.0, np.cos(angle / 2))
    p, nrm, _ = _deform(s["mesh"], k)
    for r in members:
        r.update_instance_transforms(t, first)
        r.update_mesh_vertices(p, nrm)
        r.update_top_level_acceleration_structure_async()


def test_life_after_replication(ggx_lut):
    """8 animated frames, then a texture rebind and a fresh async build on a destination: the replicated group keeps
    rendering what the directly loaded group renders."""
    s = _config4_textured(W, H)
    gs = _Groups(ggx_lut, s, "async", [0] * 3, 0)
    try:
        for k in range(1, 9):
            for members, g in ((gs.direct, gs.gd), (gs.rep, gs.gr)):
                _animate(members, s, k)
                g.frame(_params(s, members, "async"))
            _assert_equal(_capture(gs.gr, True) | _masks(gs.gr), _capture(gs.gd, True) | _masks(gs.gd), f"animated frame {k}")
        new = scenes.procedural_textures(64, seed=7)[0]
        for members, g in ((gs.direct, gs.gd), (gs.rep, gs.gr)):
            members[2].set_texture_async(0, new["levels"][0], True)
            members[1].build_acceleration_structures_async()
            g.frame(_params(s, members, "async"))
        _assert_equal(_capture(gs.gr, True) | _masks(gs.gr), _capture(gs.gd, True) | _masks(gs.gd), "rebind + rebuild")
        assert gs.rep[2].read_texture_level(0, 0).shape == (64, 64, 4)
    finally:
        gs.close()


# ---------------------------------------------------------------------------------------------------------- 4
def _moved(s, seed):
    """Scene `s` with the instances shuffled and the lights moved: the same buffer sizes, another frame."""
    t = dict(s)
    rng = np.random.default_rng(seed)
    t["instances"] = s["instances"][rng.permutation(len(s["instances"]))].copy()
    t["instances"]["translation_and_scale"][:, 1] += np.float32(0.7)
    lights = s["lights"].copy()
    lights["position_and_spotlight_epsilon"][:, 0] += np.float32(3.0)
    t["lights"] = lights
    return t


def _direct_frame(lut, s, n):
    members = [Renderer(W, H) for _ in range(n)]
    try:
        for r in members:
            _upload_scene(r, lut, s)
        with RendererGroup(members) as g:
            g.frame(s["camera"].frame_params(host.default_tonemap_params()))
            return g.read_srgb8()
    finally:
        for r in members:
            r.close()


def test_frame_before_reads_old_scene(ggx_lut):
    """Every stream held up; a group frame of scene A is enqueued with its bands read back asynchronously, then the source
    takes scene B (instances and lights) and replicates it, then a second frame: the first shows A, the second B."""
    import torch
    n = 3
    a = scenes.instanced_scene(W, H, n_instances=2000)
    b = _moved(a, 5)
    want_a, want_b = _direct_frame(ggx_lut, a, n), _direct_frame(ggx_lut, b, n)
    assert (want_a != want_b).any()
    streams = [torch.cuda.Stream(device=0) for _ in range(n)]
    members = [Renderer(W, H) for _ in range(n)]
    try:
        for r, st in zip(members, streams):
            _upload_scene(r, ggx_lut, a)
            r.set_stream(st.cuda_stream)
        fp = a["camera"].frame_params(host.default_tonemap_params())
        with RendererGroup(members) as g:
            g.frame(fp)
            g.sync()
            keep, out_a = _pinned(np.zeros((H, W, 4), np.uint8))
            for st in streams:
                _hold(st, 0.1)
            g.frame(fp)
            for r in members:
                r.read_srgb8_async(out_a)
            members[0].set_instances(b["instances"])
            members[0].set_lights(b["lights"])
            g.replicate_scene(0)
            g.frame(fp)
            got_b = g.read_srgb8()
            for r in members:
                r.wait_readback()
        for r in members:
            r.set_stream(None)
    finally:
        for r in members:
            r.close()
    assert out_a.tobytes() == want_a.tobytes(), "the frame enqueued before the call does not show the old scene"
    assert got_b.tobytes() == want_b.tobytes(), "the frame after the call does not show the replicated scene"
    del keep


def test_source_uploads_after_the_call_do_not_reach_destinations(ggx_lut):
    """The destinations' streams held up, so their copies are still queued when the source takes new instances and a new
    mesh: the destinations keep what the source held at the call."""
    import torch
    n = 3
    a = scenes.instanced_scene(W, H, n_instances=2000)
    b = _moved(a, 9)
    _, _, b["mesh"] = _deform(a["mesh"], 3, amp=0.2)
    fp = a["camera"].frame_params(host.default_tonemap_params())
    direct = [Renderer(W, H) for _ in range(n)]
    members = [Renderer(W, H) for _ in range(n)]
    streams = [torch.cuda.Stream(device=0) for _ in range(n)]
    try:
        for r in direct:
            _upload_scene(r, ggx_lut, a)
        with RendererGroup(direct) as gd:
            gd.frame(fp)
            want = _capture(gd, False)
            want_spheres = direct[1].read_chunk_spheres()
        for r, st in zip(members, streams):
            r.set_stream(st.cuda_stream)
        _upload_scene(members[0], ggx_lut, a)
        with RendererGroup(members) as g:
            g.sync()
            for st in streams[1:]:
                _hold(st, 0.1)
            g.replicate_scene(0)
            m = b["mesh"]
            members[0].set_instances(b["instances"])
            members[0].set_mesh(m["positions"], m["normals"], m["uvs"], m["indices"])
            for r in members[1:]:
                assert r.read_chunk_spheres().tobytes() == want_spheres.tobytes(), "a destination received the later mesh"
            m = a["mesh"]   # the source back to scene A: the whole group frame must then be A's
            members[0].set_instances(a["instances"])
            members[0].set_mesh(m["positions"], m["normals"], m["uvs"], m["indices"])
            g.frame(fp)
            _assert_equal(_capture(g, False), want, "after later uploads to the source")
        for r in members:
            r.set_stream(None)
    finally:
        for r in direct + members:
            r.close()


def test_replicate_does_not_block(ggx_lut):
    """With the source stream held up for 0.2 s, the call returns at once once the destinations' buffers have their size."""
    import torch
    s = _config4_textured(W, H)
    stream = torch.cuda.Stream(device=0)
    keep = {}
    members = [Renderer(W, H) for _ in range(3)]
    try:
        members[0].set_stream(stream.cuda_stream)
        _load(members[0], ggx_lut, s, "async", keep)
        with RendererGroup(members) as g:
            g.replicate_scene(0)   # sizes every destination buffer
            g.sync()
            _hold(stream, 0.2)
            t0 = time.perf_counter()
            g.replicate_scene(0)
            call = time.perf_counter() - t0
            g.sync()
            total = time.perf_counter() - t0
        members[0].set_stream(None)
    finally:
        for r in members:
            r.close()
    print(f"tr_group_replicate_scene returned after {call * 1e3:.2f} ms; the copies finished after {total * 1e3:.1f} ms")
    assert total > 0.15, "the sleep did not hold up the source stream"
    assert call < 0.1, f"tr_group_replicate_scene blocked for {call * 1e3:.1f} ms"


# ---------------------------------------------------------------------------------------------------------- 5
def _replicate_status(g, source):
    out = (C.c_uint64 * 8)()
    st = _lib().tr_group_replicate_scene(g._g, C.c_uint32(source), out)
    return st, _lib().tr_last_error().decode()


def test_rules(ggx_lut):
    s = _config4_textured(W, H)
    keep = {}
    a, b, c = (Renderer(W, H) for _ in range(3))
    lone = Renderer(W, H)
    groups = []
    try:
        _load(a, ggx_lut, s, "host", keep)
        _load(c, ggx_lut, s, "async", keep)   # c: its own structures, whose handle goes stale below
        stale = c.acceleration_structure_address
        g = RendererGroup([a, b, c])
        groups.append(g)
        before = [_state(a, s, "host"), _state(c, s, "async")]
        for source, status, words in ((3, TR_ERR_INVALID_ARG, "source 3"), (1, TR_ERR_STATE, "no mesh")):
            n0 = Renderer.launch_count()
            st, msg = _replicate_status(g, source)
            assert st == status and words in msg, (source, st, msg)
            assert Renderer.launch_count() == n0
        _assert_equal(_state(a, s, "host"), before[0], "a rejected call changed member 0")
        _assert_equal(_state(c, s, "async"), before[1], "a rejected call changed member 2")
        assert len(b.read_chunk_spheres()) == 0, "a rejected call gave member 1 a mesh"

        g.sync()
        own = a.acceleration_structure_address   # the source's handle from its own build
        n0 = Renderer.launch_count()
        addresses = g.replicate_scene(0)
        assert Renderer.launch_count() == n0, "the call launched a kernel"
        assert addresses[0] == own and all(addresses) and len(set(addresses)) == 3, (own, addresses)
        g.frame(_params(s, [a, b, c], "host"))   # every member's returned handle is accepted
        g.sync()

        # a source without structures: every handle is 0, and one a destination built itself is refused
        b.set_mesh(s["mesh"]["positions"], s["mesh"]["normals"], s["mesh"]["uvs"], s["mesh"]["indices"])   # drops b's trees
        assert g.replicate_scene(1) == [0, 0, 0]
        bad = _params(s, [a, b, c], "none")
        bad[2]["push_constants"]["acceleration_structure_address"] = stale
        with pytest.raises(TrError) as e:
            g.frame(bad)
        assert e.value.status == TR_ERR_INVALID_ARG
        g.frame(_params(s, [a, b, c], "none"))
        g.sync()

        # a group of one copies nothing
        _load(lone, ggx_lut, s, "async", keep)
        own = lone.acceleration_structure_address
        with RendererGroup([lone]) as one:
            state = _state(lone, s, "async")
            n0 = Renderer.launch_count()
            assert one.replicate_scene(0) == [own] and own != 0
            assert Renderer.launch_count() == n0
            _assert_equal(_state(lone, s, "async"), state, "group of one")
            one.frame(_params(s, [lone], "async"))   # the returned handle is accepted
            one.sync()
            st, msg = _replicate_status(one, 1)
            assert st == TR_ERR_INVALID_ARG, msg
    finally:
        for g in groups:
            g.close()
        for r in (a, b, c, lone):
            r.close()


# ---------------------------------------------------------------------------------------------------------- 6
@pytest.mark.parametrize("n", [2, 4])
def test_members_on_one_device(ggx_lut, n):
    """2 and 4 members on device 0, the last one the source, async structures."""
    s = _config4_textured(W, H)
    gs = _Groups(ggx_lut, s, "async", [0] * n, n - 1)
    try:
        gs.gd.frame(_params(s, gs.direct, "async"))
        gs.gr.frame(_params(s, gs.rep, "async"))
        _assert_equal(_capture(gs.gr, True) | _masks(gs.gr), _capture(gs.gd, True) | _masks(gs.gd), f"{n} members")
    finally:
        gs.close()


def test_across_devices(ggx_lut):
    import torch
    n_dev = torch.cuda.device_count()
    if n_dev < 2:
        pytest.skip(f"{n_dev} GPU visible: replication across devices needs at least 2")
    s = _config4_textured(W, H)
    for devices, rt in ((list(range(min(8, n_dev))), "async"), ([d for d in range(min(2, n_dev)) for _ in range(2)], "host")):
        gs = _Groups(ggx_lut, s, rt, devices, len(devices) - 1)
        try:
            gs.gd.frame(_params(s, gs.direct, rt))
            gs.gr.frame(_params(s, gs.rep, rt))
            _assert_equal(_capture(gs.gr, True) | _masks(gs.gr), _capture(gs.gd, True) | _masks(gs.gd), f"devices {devices}")
            ref = _state(gs.rep[-1], s, rt)
            for k, r in enumerate(gs.rep[:-1]):
                _assert_equal(_state(r, s, rt), ref, f"devices {devices}: member {k}'s state")
        finally:
            gs.close()
