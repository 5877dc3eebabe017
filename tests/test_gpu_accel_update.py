"""tr_update_top_level_acceleration_structure_async: the top level rebuilt on the device in stream order (k_accel_device.cu,
a linear BVH) against the host's binned-SAH update.  The trees differ; the occlusion result is defined without them
(DESIGN.md section 7 N4), so rays, shadow masks and frames must agree bit for bit, and the instance records byte for byte."""
import time

import numpy as np
import pytest

from accel_checks import ACCEL_STACK, ASYNC_TLAS_LAUNCHES as ASYNC_UPDATE_LAUNCHES
from accel_checks import _hold, _pinned, _random_rays, _reference, _surface_rays, _tree_checks, _upload_scene
from pipeline import REL_L2_TOL, rel_l2
from transmission_renderer_b200 import Renderer, RendererGroup, TrError, abi, host, scenes

pytestmark = pytest.mark.gpu
f32 = np.float32
TR_ERR_INVALID_ARG, TR_ERR_STATE = -1, -6


def _same_records(a, b):
    ra = np.sort(np.frombuffer(a.tobytes(), np.dtype((np.void, 64))))
    rb = np.sort(np.frombuffer(b.tobytes(), np.dtype((np.void, 64))))
    return len(ra) == len(rb) and ra.tobytes() == rb.tobytes()


def _host_and_async(r, instances):
    """The same instances through both updates of one context: (host tree, async tree) as (nodes, records)."""
    r.set_instances(instances)
    h = r.update_top_level_acceleration_structure()
    host_tree = r.read_top_level_acceleration_structure()
    r.set_instances(instances)
    a = r.update_top_level_acceleration_structure_async()
    assert a == h
    return host_tree, r.read_top_level_acceleration_structure()


@pytest.mark.parametrize("kind", ["shadow", "instanced"])
def test_rays_and_records_bit_exact(oracle, ggx_lut, kind):
    w, h = 320, 180
    s = scenes.shadow_scene(w, h) if kind == "shadow" else scenes.instanced_scene(w, h, n_instances=2000, n_lights=16)
    acc = oracle.Accel(s["mesh"], s["instances"], s["primitives"])
    rng = np.random.default_rng(17)
    box = ([-8, 0, -10], [8, 6, 6]) if kind == "shadow" else ([-30, 0, -30], [30, 12, 30])
    o, d, t = _random_rays(rng, 200000, *box)
    po, pd, pt = _surface_rays(s, oracle, 100000, rng)
    with Renderer(w, h) as r:
        _upload_scene(r, ggx_lut, s)
        r.build_acceleration_structures()
        host_rays = r.trace_shadow_rays(o, d, t), r.trace_shadow_rays(po, pd, pt)
        (hn, hi), (an, ai) = _host_and_async(r, s["instances"])
        async_rays = r.trace_shadow_rays(o, d, t), r.trace_shadow_rays(po, pd, pt)
    ref = acc.trace(o, d, t), acc.trace(po, pd, pt)
    for got_h, got_a, want in zip(host_rays, async_rays, ref):
        assert (got_a != want).sum() == 0 and (got_h != want).sum() == 0
    assert 0.02 < 1 - ref[0].mean() < 0.98 and 0.02 < 1 - ref[1].mean() < 0.98
    sub = slice(0, 20000)
    assert np.array_equal(async_rays[0][sub], acc.trace(o[sub], d[sub], t[sub], brute=True))
    # records: the host's bytes, as a multiset; the tree: exact unions, every instance once, bounded depth
    n_top = int(sum(1 for p in s["instances"]["primitive_id"] if s["primitives"]["draw_buffer_index"][p] < 2))
    assert len(ai) == len(hi) == n_top and len(an) == len(hn) == max(n_top - 1, 1)
    assert _same_records(ai, hi)
    depth = _tree_checks(an, ai)
    _tree_checks(hn, hi)
    print(f"{kind}: {n_top} top-level instances, LBVH depth {depth}")
    assert depth < ACCEL_STACK


def _quat(axis, angle):
    axis = np.asarray(axis, np.float64)
    axis = axis / np.linalg.norm(axis)
    return np.concatenate([axis * np.sin(angle / 2), [np.cos(angle / 2)]])


def _pathological(s):
    """name -> instances over shadow_scene's primitives (0 sphere, 1 box, 2 quad, 3 alpha-clip sphere, 4 glass knot)."""
    rng = np.random.default_rng(5)
    out = {}
    same = np.zeros(4096, abi.instance)            # one centroid: every Morton code equal
    same["translation_and_scale"] = (0.5, 1.0, -1.0, 0.8)
    same["rotation"] = (0.0, 0.0, 0.0, 1.0)
    same["primitive_id"] = 1
    out["one_centroid"] = same
    n = 48                                          # a chain at geometrically shrinking offsets
    chain = np.zeros(n, abi.instance)
    off = 3.0 * 0.5 ** np.arange(n)
    chain["translation_and_scale"][:, 0] = -1.5 + off
    chain["translation_and_scale"][:, 1] = 1.0 + 0.5 * off
    chain["translation_and_scale"][:, 2] = -1.0
    chain["translation_and_scale"][:, 3] = 0.15
    chain["rotation"] = [_quat((1, 2, 3), 0.3 * k) for k in range(n)]
    chain["primitive_id"] = np.arange(n) % 2
    out["chain"] = chain
    n = 300                                         # scales over five decades, zero and negative
    sc = np.zeros(n, abi.instance)
    sc["translation_and_scale"][:, :3] = rng.uniform((-6, 0, -8), (6, 4, 4), (n, 3))
    mag = 10.0 ** rng.uniform(-3, 2, n)
    mag[::17] = 0.0
    sc["translation_and_scale"][:, 3] = mag * np.where(rng.random(n) < 0.3, -1.0, 1.0)
    sc["rotation"] = [_quat(rng.normal(size=3), rng.uniform(0, 6.3)) for _ in range(n)]
    sc["primitive_id"] = rng.integers(0, 4, n)
    out["scales"] = sc
    glass = s["instances"][s["instances"]["primitive_id"] == 4]
    out["none_cast"] = np.concatenate([glass, glass])   # only the transmissive knot: m = 0
    one = s["instances"][s["instances"]["primitive_id"] == 0][:1].copy()
    out["single"] = np.concatenate([one, glass])        # m = 1
    return out


@pytest.mark.parametrize("case", ["one_centroid", "chain", "scales", "none_cast", "single"])
def test_pathological_inputs(oracle, ggx_lut, case):
    w, h = 160, 90
    s = scenes.shadow_scene(w, h)
    inst = _pathological(s)[case]
    rng = np.random.default_rng(23)
    o, d, t = _random_rays(rng, 6000, [-8, 0, -10], [8, 6, 6])
    n_rays = 1500 if case == "one_centroid" else len(o)
    o, d, t = o[:n_rays], d[:n_rays], t[:n_rays]
    with Renderer(w, h) as r:
        _upload_scene(r, ggx_lut, s)
        r.build_acceleration_structures()
        (hn, hi), (an, ai) = _host_and_async(r, inst)
        got_async = r.trace_shadow_rays(o, d, t)
        r.update_top_level_acceleration_structure()
        got_host = r.trace_shadow_rays(o, d, t)
    acc = oracle.Accel(s["mesh"], inst, s["primitives"])
    brute = acc.trace(o, d, t, brute=True)
    assert np.array_equal(got_async, brute), f"{(got_async != brute).sum()} rays differ from the definition"
    assert np.array_equal(got_host, brute)
    assert _same_records(ai, hi)
    depth = _tree_checks(an, ai)
    print(f"{case}: m = {len(ai)}, LBVH depth {depth}, occluded {1 - brute.mean():.3f}")
    assert depth < ACCEL_STACK
    want_m = {"none_cast": 0, "single": 1}.get(case)
    if want_m is not None:
        assert len(ai) == want_m and len(an) == 1


def _rotated_frames(instances, n_frames):
    """Every instance turned a little more each frame (the reference's --rotate-model, applied to all of them)."""
    out = []
    q = instances["rotation"].astype(np.float64)
    for f in range(n_frames):
        step = _quat((0.3, 1.0, 0.2), 0.04 * (f + 1))
        x1, y1, z1, w1 = step
        x2, y2, z2, w2 = q.T
        r = np.stack([w1 * x2 + x1 * w2 + y1 * z2 - z1 * y2, w1 * y2 - x1 * z2 + y1 * w2 + z1 * x2,
                      w1 * z2 + x1 * y2 - y1 * x2 + z1 * w2, w1 * w2 - x1 * x2 - y1 * y2 - z1 * z2], 1)
        inst = instances.copy()
        inst["rotation"] = r.astype(f32)
        out.append(inst)
    return out


def test_animation_matches_host_update(oracle, ggx_lut):
    """8 frames in which every instance rotates: async update (pinned uploads, no sync between frames) against the host
    update, masks of both layers, HDR and sRGB8 equal frame by frame; the last frame against the oracle."""
    w, h = 480, 270
    s = scenes.shadow_scene(w, h)
    cam = s["camera"]
    frames = _rotated_frames(s["instances"], 8)
    keep = [_pinned(f) for f in frames]
    tm = host.default_tonemap_params()

    def outputs(r):
        return r.read_shadow_mask(0), r.read_shadow_mask(1), r.read_hdr(), r.read_srgb8()

    with Renderer(w, h, f32_debug=True) as r:
        _upload_scene(r, ggx_lut, s)
        r.build_acceleration_structures()
        want = []
        for inst in frames:
            r.set_instances(inst)
            hdl = r.update_top_level_acceleration_structure()
            r.frame(cam.frame_params(tm, acceleration_structure_address=hdl))
            want.append(outputs(r))
    with Renderer(w, h, f32_debug=True) as r:
        _upload_scene(r, ggx_lut, s)
        handle = r.build_acceleration_structures()
        for k, (_, pin) in enumerate(keep):
            r.set_instances(pin)
            assert r.update_top_level_acceleration_structure_async() == handle
            r.frame(cam.frame_params(tm, acceleration_structure_address=handle))
            got = outputs(r)
            for name, a, b in zip(("opaque mask", "transmissive mask", "HDR", "sRGB8"), got, want[k]):
                assert a.tobytes() == b.tobytes(), f"frame {k}: {name} differs"
        last32 = r.read_hdr_f32()
        for _, pin in keep:                 # again, back to back: nothing read until the end
            r.set_instances(pin)
            r.update_top_level_acceleration_structure_async()
            r.frame(cam.frame_params(tm, acceleration_structure_address=handle))
        r.sync()
        got = outputs(r)
    for name, a, b in zip(("opaque mask", "transmissive mask", "HDR", "sRGB8"), got, want[-1]):
        assert a.tobytes() == b.tobytes(), f"back to back: {name} differs"
    assert (want[0][0] != want[-1][0]).any(0).mean() > 0.005, "the animation does not move the shadows"
    s2 = dict(s, instances=frames[-1])
    ref = _reference(oracle, ggx_lut, s2, oracle.Accel(s2["mesh"], s2["instances"], s2["primitives"]))
    assert (want[-1][0] != oracle.shadow_mask_frame(ref["g0"], ref["scene"])).sum() == 0
    assert rel_l2(last32[..., :3], ref["t32"][..., :3]) < REL_L2_TOL


def test_async_update_does_not_block(ggx_lut):
    """With the context's stream held up on the GPU, set_instances (page-locked) + the async update + frame return at
    once; the host update in the same place waits for the GPU."""
    import torch
    w, h = 960, 540
    s = scenes.instanced_scene(w, h, n_instances=4000, n_lights=32)
    fp = lambda hdl: s["camera"].frame_params(host.default_tonemap_params(), acceleration_structure_address=hdl)
    frames = _rotated_frames(s["instances"], 3)
    keep = [_pinned(f) for f in frames]
    stream = torch.cuda.Stream(device=0)
    with Renderer(w, h) as r:
        r.set_stream(stream.cuda_stream)
        _upload_scene(r, ggx_lut, s)
        handle = r.build_acceleration_structures()
        for _, pin in keep[:2]:            # warm-up: the primitive table, the builder's scratch, the frame buffers
            r.set_instances(pin)
            r.update_top_level_acceleration_structure_async()
            r.frame(fp(handle))
        r.sync()
        _hold(stream, 0.2)
        t0 = time.perf_counter()
        r.set_instances(keep[2][1])
        r.update_top_level_acceleration_structure_async()
        r.frame(fp(handle))
        enqueue = time.perf_counter() - t0
        r.sync()
        total = time.perf_counter() - t0
        _hold(stream, 0.2)
        t0 = time.perf_counter()
        r.set_instances(keep[1][1])
        r.update_top_level_acceleration_structure()
        blocking = time.perf_counter() - t0
        r.sync()
        r.set_stream(None)
    print(f"async: enqueue {enqueue * 1e3:.1f} ms, frame done after {total * 1e3:.1f} ms; host update {blocking * 1e3:.1f} ms")
    assert total > 0.15, "the sleep did not hold up the stream"
    assert enqueue < 0.1, f"set_instances + async update + frame blocked for {enqueue * 1e3:.1f} ms"
    assert blocking > 0.15


def test_group_with_async_updates(ggx_lut):
    """3 members on one device, each updated on the device before tr_group_frame: the frame equals one context's (host
    update) bit for bit, and the whole enqueue stays non-blocking while member 0's stream is held up."""
    import torch
    w, h = 960, 540
    s = scenes.shadow_scene(w, h)
    cam = s["camera"]
    tm = host.default_tonemap_params()
    frames = _rotated_frames(s["instances"], 3)
    keep = [_pinned(f) for f in frames]
    with Renderer(w, h) as r:
        _upload_scene(r, ggx_lut, s)
        r.build_acceleration_structures()
        r.set_instances(frames[-1])
        r.frame(cam.frame_params(tm, acceleration_structure_address=r.update_top_level_acceleration_structure()))
        want = r.read_hdr(), r.read_srgb8()
    stream = torch.cuda.Stream(device=0)
    members = [Renderer(w, h) for _ in range(3)]
    try:
        members[0].set_stream(stream.cuda_stream)
        for r in members:
            _upload_scene(r, ggx_lut, s)
            r.build_acceleration_structures()
        with RendererGroup(members) as g:
            for _, pin in keep[:2]:          # warm-up
                for r in members:
                    r.set_instances(pin)
                    r.update_top_level_acceleration_structure_async()
                g.frame(cam.frame_params(tm, acceleration_structure_address=1))
            g.sync()
            _hold(stream, 0.2)
            t0 = time.perf_counter()
            for r in members:
                r.set_instances(keep[2][1])
                r.update_top_level_acceleration_structure_async()
            g.frame(cam.frame_params(tm, acceleration_structure_address=1))   # each member's own handle goes in
            enqueue = time.perf_counter() - t0
            g.sync()
            total = time.perf_counter() - t0
            got = g.read_hdr(), g.read_srgb8()
        members[0].set_stream(None)
    finally:
        for r in members:
            r.close()
    print(f"group: enqueue {enqueue * 1e3:.1f} ms, frame done after {total * 1e3:.1f} ms")
    assert got[0].tobytes() == want[0].tobytes(), "group HDR differs from one context"
    assert got[1].tobytes() == want[1].tobytes(), "group sRGB8 differs from one context"
    assert total > 0.15, "the sleep did not hold up member 0's stream"
    assert enqueue < 0.1, f"per-member async updates + tr_group_frame blocked for {enqueue * 1e3:.1f} ms"


def test_rules(ggx_lut):
    w, h = 160, 90
    s = scenes.shadow_scene(w, h)
    cam = s["camera"]
    with Renderer(w, h) as r:
        _upload_scene(r, ggx_lut, s)
        with pytest.raises(TrError) as e:
            r.update_top_level_acceleration_structure_async()               # before tr_build_acceleration_structures
        assert e.value.status == TR_ERR_STATE
        handle = r.build_acceleration_structures()
        assert r.update_top_level_acceleration_structure_async() == handle  # first call: uploads the primitive table
        r.sync()
        before = Renderer.launch_count()
        assert r.update_top_level_acceleration_structure_async() == handle  # same m: same handle
        assert Renderer.launch_count() - before == ASYNC_UPDATE_LAUNCHES
        r.frame(cam.frame_params(acceleration_structure_address=handle))
        # an instance naming a missing primitive: refused before anything is enqueued
        bad = s["instances"].copy()
        bad["primitive_id"][3] = 99
        r.set_instances(bad)
        r.sync()
        before = Renderer.launch_count()
        with pytest.raises(TrError) as e:
            r.update_top_level_acceleration_structure_async()
        assert e.value.status == TR_ERR_INVALID_ARG and "instance 3" in str(e.value)
        assert Renderer.launch_count() == before
        # set_instances without an update: the next traced frame is refused
        r.set_instances(s["instances"])
        with pytest.raises(TrError) as e:
            r.frame(cam.frame_params(acceleration_structure_address=handle))
        assert e.value.status == TR_ERR_STATE
        assert r.update_top_level_acceleration_structure_async() == handle
        r.frame(cam.frame_params(acceleration_structure_address=handle))
        # rebinding the mesh invalidates the handle and the update
        m = s["mesh"]
        r.set_mesh(m["positions"], m["normals"], m["uvs"], m["indices"])
        with pytest.raises(TrError):
            r.frame(cam.frame_params(acceleration_structure_address=handle))
        with pytest.raises(TrError) as e:
            r.update_top_level_acceleration_structure_async()
        assert e.value.status == TR_ERR_STATE
        r.sync()
