"""tr_update_mesh_vertices: vertex animation in stream order.  The culling spheres of the binning pass are recomputed on the
device (byte for byte the formula restated below), and the bottom-level trees are refitted: same topology, new triangles and
boxes.  The occlusion result is defined without the trees (DESIGN.md section 7 N4), so a context that was updated must render
and trace exactly what a fresh context renders and traces after tr_set_mesh + tr_build_acceleration_structures with the same
final arrays."""
import time

import numpy as np
import pytest

from accel_checks import MESH_UPDATE_LAUNCHES, MESH_UPDATE_LAUNCHES_NO_ACCEL
from accel_checks import _check_blas, _deform, _hold, _pinned, _random_rays, _records_key, _reference, _surface_rays, _upload_scene
from pipeline import REL_L2_TOL, rel_l2
from transmission_renderer_b200 import Renderer, RendererGroup, TrError, abi, host, scenes

pytestmark = pytest.mark.gpu
f32 = np.float32
TR_ERR_INVALID_ARG, TR_ERR_STATE = -1, -6
CHUNK = 64                     # TR_CHUNK_TRIS


# ---------------------------------------------------------------------------------------------------------- restatements
def _fold_first(vals, better, init):
    """Sequential `acc = better(v, acc) ? v : acc` from `init`: NaN never wins, and of two equal extremes (-0, +0) the first
    stays."""
    acc = init
    ok = ~np.isnan(vals) & better(vals, init)
    if ok.any():
        cand = vals[ok]
        m = cand.min() if better(-1.0, 1.0) else cand.max()
        acc = cand[np.nonzero(cand == m)[0][0]]
    return float(acc)


def _chunk_spheres(pos, idx, prims):
    """ensure_chunks in numpy: per 64 triangles, the box in double, centre 0.5 (lo + hi), farthest vertex in double, the
    radius widened by the centre's rounding to float and by 1 + 1e-6; infinity when that is not finite."""
    out = []
    with np.errstate(all="ignore"):
        for p in prims:
            first, tris = int(p["first_index"]), int(p["index_count"]) // 3
            for t0 in range(0, tris, CHUNK):
                t1 = min(t0 + CHUNK, tris)
                v = pos[idx[first + t0 * 3:first + t1 * 3]].astype(np.float64)
                lo = [_fold_first(v[:, k], lambda a, b: np.less(a, b), 1e300) for k in range(3)]
                hi = [_fold_first(v[:, k], lambda a, b: np.greater(a, b), -1e300) for k in range(3)]
                c = [0.5 * (lo[k] + hi[k]) for k in range(3)]
                d = v - np.array(c)
                sq = (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]
                sq = sq[~np.isnan(sq)]
                r2 = max(0.0, float(sq.max())) if len(sq) else 0.0
                fc = [f32(x) for x in c]
                shift = (abs(float(fc[0]) - c[0]) + abs(float(fc[1]) - c[1])) + abs(float(fc[2]) - c[2])
                r = f32((np.sqrt(r2) + shift) * (1.0 + 1e-6))
                if not np.isfinite(r):
                    r = f32(np.inf)
                out.append((fc[0], fc[1], fc[2], r))
    return np.array(out, f32).reshape(-1, 4)


def _vertex_ranges(s):
    """[first vertex, end) of every primitive of a MeshSet scene (from its index ranges)."""
    idx = s["mesh"]["indices"]
    out = []
    for p in s["primitives"]:
        sl = idx[int(p["first_index"]):int(p["first_index"]) + int(p["index_count"])]
        out.append((int(sl.min()), int(sl.max()) + 1))
    return out


def _fresh(w, h, lut, s, mesh, accel=True, f32_debug=False):
    r = Renderer(w, h, f32_debug=f32_debug)
    _upload_scene(r, lut, dict(s, mesh=mesh))
    handle = r.build_acceleration_structures() if accel else 0
    return r, handle


# ---------------------------------------------------------------------------------------------------------- 1. chunk spheres
@pytest.mark.parametrize("kind", ["shadow", "instanced"])
def test_chunk_spheres_byte_equal(ggx_lut, kind):
    w, h = 160, 90
    s = scenes.shadow_scene(w, h) if kind == "shadow" else scenes.instanced_scene(w, h, n_instances=500, n_lights=8)
    m = s["mesh"]
    with Renderer(w, h) as r:
        _upload_scene(r, ggx_lut, s)
        got = r.read_chunk_spheres()
        want = _chunk_spheres(m["positions"], m["indices"], s["primitives"])
        assert len(got) == len(want) > 0 and got.tobytes() == want.tobytes()
        r.frame(s["camera"].frame_params(host.default_tonemap_params()))
        mesh = m
        ranges = _vertex_ranges(s)
        for k, (a, b) in enumerate([(0, None), ranges[-1], (ranges[1][0] + 7, ranges[2][0] + 11)]):
            pos, nrm, mesh = _deform(mesh, k + 1, a, b)
            r.update_mesh_vertices(pos, nrm, first_vertex=a)
            got = r.read_chunk_spheres()
            want = _chunk_spheres(mesh["positions"], mesh["indices"], s["primitives"])
            assert got.tobytes() == want.tobytes(), f"update {k}: {(got != want).any(1).sum()} spheres differ"


def _extreme_mesh():
    """Two primitives, 130 and 77 triangles (not multiples of 64), with degenerate triangles, signed zeros, coordinates
    around 1e30, and one chunk with an infinite and a NaN vertex."""
    rng = np.random.default_rng(3)
    nv = 300
    pos = rng.normal(size=(nv, 3)).astype(f32)
    pos[10:20] = 0.0
    pos[12:16, 1] = -0.0
    pos[40:60] = (rng.normal(size=(20, 3)) * 1e30).astype(f32)
    idx = rng.integers(0, nv, (207, 3)).astype(np.uint32)
    idx[5] = (10, 10, 10)                  # degenerate: one vertex
    idx[6] = (11, 12, 11)
    idx[7:9] = (13, 14, 15)
    idx[100:110, 0] = rng.integers(40, 60, 10)
    idx[150] = (250, 251, 252)
    pos[251] = (np.inf, 1.0, 2.0)
    pos[252, 2] = np.nan
    prims = np.zeros(2, abi.primitive_info)
    prims["index_count"] = (130 * 3, 77 * 3)
    prims["first_index"] = (0, 130 * 3)
    prims["packed_bounding_sphere"] = (0.0, 0.0, 0.0, 1e38)
    return pos, idx.reshape(-1), prims


def test_chunk_spheres_extreme_inputs():
    pos, idx, prims = _extreme_mesh()
    nrm = np.tile(np.array([0.0, 1.0, 0.0], f32), (len(pos), 1))
    uv = np.zeros((len(pos), 2), f32)
    with Renderer(64, 64) as r:
        r.set_primitives(prims)
        r.set_mesh(pos, nrm, uv, idx)
        got = r.read_chunk_spheres()
        want = _chunk_spheres(pos, idx, prims)
        assert len(got) == 3 + 2
        assert got.tobytes() == want.tobytes()
        assert np.isinf(want[:, 3]).any() and np.isfinite(want[:, 3]).any()
        new = pos.copy()                    # a partial range: a zero turned negative, a huge vertex, the infinity gone
        new[11:260] = new[11:260][::-1]
        new[30] = (-0.0, 5e29, -0.0)
        r.update_mesh_vertices(new[11:260], nrm[11:260], first_vertex=11)
        got = r.read_chunk_spheres()
        want = _chunk_spheres(new, idx, prims)
        assert got.tobytes() == want.tobytes(), f"{(got.view(np.uint32) != want.view(np.uint32)).any(1).sum()} spheres differ"


# ---------------------------------------------------------------------------------------------------------- 2. raster path
def test_raster_path_matches_fresh_context(oracle, ggx_lut):
    """Deformations with ray queries off, some of them partial ranges: G-buffer planes, HDR and sRGB8 equal to a fresh
    context's; the last frame against the oracle."""
    w, h = 480, 270
    s = scenes.shadow_scene(w, h)
    cam = s["camera"]
    tm = host.default_tonemap_params()
    ranges = _vertex_ranges(s)
    steps = [(0, None), ranges[4], (ranges[0][0] + 100, ranges[3][0] + 50), ranges[1], (0, None)]
    fresh = Renderer(w, h, f32_debug=True)
    try:
        _upload_scene(fresh, ggx_lut, s)
        with Renderer(w, h, f32_debug=True) as r:
            _upload_scene(r, ggx_lut, s)
            r.frame(cam.frame_params(tm))
            mesh = s["mesh"]
            for k, (a, b) in enumerate(steps):
                pos, nrm, mesh = _deform(mesh, k + 1, a, b)
                r.update_mesh_vertices(pos, nrm, first_vertex=a)
                r.frame(cam.frame_params(tm))
                fresh.set_mesh(mesh["positions"], mesh["normals"], mesh["uvs"], mesh["indices"])
                fresh.frame(cam.frame_params(tm))
                for layer in (0, 1):
                    g, gw = r.read_gbuffer(layer), fresh.read_gbuffer(layer)
                    for name in ("depth", "normal", "uv", "material_id", "scale"):
                        assert g[name].tobytes() == gw[name].tobytes(), f"step {k}: layer {layer} {name} differs"
                assert r.read_hdr().tobytes() == fresh.read_hdr().tobytes(), f"step {k}: HDR differs"
                assert r.read_srgb8().tobytes() == fresh.read_srgb8().tobytes(), f"step {k}: sRGB8 differs"
            last32 = r.read_hdr_f32()
    finally:
        fresh.close()
    assert not np.array_equal(mesh["positions"], s["mesh"]["positions"])
    ref = _reference(oracle, ggx_lut, dict(s, mesh=mesh), None)
    e = rel_l2(last32[..., :3], ref["t32"][..., :3])
    print(f"raster path after {len(steps)} updates: rel-L2 {e:.2e} against the oracle")
    assert e < REL_L2_TOL


# ---------------------------------------------------------------------------------------------------------- 3. refit
@pytest.mark.parametrize("kind", ["shadow", "instanced"])
def test_refit(oracle, ggx_lut, kind):
    w, h = 320, 180
    s = scenes.shadow_scene(w, h) if kind == "shadow" else scenes.instanced_scene(w, h, n_instances=2000, n_lights=16)
    rng = np.random.default_rng(29)
    box = ([-8, 0, -10], [8, 6, 6]) if kind == "shadow" else ([-30, 0, -30], [30, 12, 30])
    o, d, t = _random_rays(rng, 200000, *box)
    pos, nrm, mesh = _deform(s["mesh"], 3, amp=0.08)
    s2 = dict(s, mesh=mesh)
    po, pd, pt = _surface_rays(s2, oracle, 100000, rng)
    with Renderer(w, h) as r:
        _upload_scene(r, ggx_lut, s)
        handle = r.build_acceleration_structures()
        nodes0, _ = r.read_bottom_level_acceleration_structure()
        r.update_mesh_vertices(pos, nrm)
        assert r.update_top_level_acceleration_structure_async() == handle
        nodes, tris = r.read_bottom_level_acceleration_structure()
        _, inst_async = r.read_top_level_acceleration_structure()
        got = r.trace_shadow_rays(o, d, t), r.trace_shadow_rays(po, pd, pt)
        r.update_top_level_acceleration_structure()
        _, inst_host = r.read_top_level_acceleration_structure()
        got_host = r.trace_shadow_rays(o, d, t)
    fresh, _ = _fresh(w, h, ggx_lut, s, mesh)
    with fresh:
        want = fresh.trace_shadow_rays(o, d, t), fresh.trace_shadow_rays(po, pd, pt)
        _, inst_fresh = fresh.read_top_level_acceleration_structure()
    assert np.array_equal(nodes["c0"], nodes0["c0"]) and np.array_equal(nodes["c1"], nodes0["c1"]), "the topology changed"
    _check_blas(nodes, tris, s["primitives"], mesh)
    assert _records_key(inst_async).tobytes() == _records_key(inst_fresh).tobytes(), "async top level after the refit"
    assert _records_key(inst_host).tobytes() == _records_key(inst_fresh).tobytes(), "blocking top level after the refit"
    for g, wnt in zip(got, want):
        assert (g != wnt).sum() == 0, f"{(g != wnt).sum()} rays differ from the fresh context"
    assert np.array_equal(got_host, want[0])
    acc = oracle.Accel(mesh, s["instances"], s["primitives"])
    sub = slice(0, 20000)
    assert np.array_equal(got[0][sub], acc.trace(o[sub], d[sub], t[sub], brute=True))
    assert np.array_equal(got[1][sub], acc.trace(po[sub], pd[sub], pt[sub], brute=True))
    assert 0.02 < 1 - want[0].mean() < 0.98


# ---------------------------------------------------------------------------------------------------------- 4. animation
def test_animation_matches_fresh_context(oracle, ggx_lut):
    """8 deformed frames with ray queries on (page-locked sources, async top-level update): shadow masks, HDR and sRGB8
    equal to a fresh context's frame by frame; the last frame against the oracle."""
    w, h = 480, 270
    s = scenes.shadow_scene(w, h)
    cam = s["camera"]
    tm = host.default_tonemap_params()
    meshes, mesh = [], s["mesh"]
    for k in range(8):
        pos, nrm, mesh = _deform(s["mesh"], k + 1, amp=0.06)
        meshes.append((_pinned(pos), _pinned(nrm), mesh))

    def outputs(r):
        return r.read_shadow_mask(0), r.read_shadow_mask(1), r.read_hdr(), r.read_srgb8()

    fresh = Renderer(w, h, f32_debug=True)
    try:
        _upload_scene(fresh, ggx_lut, s)
        with Renderer(w, h, f32_debug=True) as r:
            _upload_scene(r, ggx_lut, s)
            handle = r.build_acceleration_structures()
            for k, ((_, pos), (_, nrm), m) in enumerate(meshes):
                r.update_mesh_vertices(pos, nrm)
                assert r.update_top_level_acceleration_structure_async() == handle
                r.frame(cam.frame_params(tm, acceleration_structure_address=handle))
                got = outputs(r)
                fresh.set_mesh(m["positions"], m["normals"], m["uvs"], m["indices"])
                fresh.frame(cam.frame_params(tm, acceleration_structure_address=fresh.build_acceleration_structures()))
                want = outputs(fresh)
                for name, a, b in zip(("opaque mask", "transmissive mask", "HDR", "sRGB8"), got, want):
                    assert a.tobytes() == b.tobytes(), f"frame {k}: {name} differs"
                if k == 0:
                    first_mask = got[0]
            last32 = r.read_hdr_f32()
    finally:
        fresh.close()
    assert (first_mask != got[0]).any(0).mean() > 0.0005, "the deformation does not move the shadows"
    s2 = dict(s, mesh=meshes[-1][2])
    ref = _reference(oracle, ggx_lut, s2, oracle.Accel(s2["mesh"], s2["instances"], s2["primitives"]))
    assert (got[0] != oracle.shadow_mask_frame(ref["g0"], ref["scene"])).sum() == 0
    assert (got[1] != oracle.shadow_mask_frame(ref["g1"], ref["scene"])).sum() == 0
    assert rel_l2(last32[..., :3], ref["t32"][..., :3]) < REL_L2_TOL


# ---------------------------------------------------------------------------------------------------------- 5. stream order
def test_stream_order(ggx_lut):
    """frame A, read-back of A, update, frame B, all enqueued before any wait: A shows the old mesh, B the new one."""
    w, h = 480, 270
    s = scenes.shadow_scene(w, h)
    cam = s["camera"]
    tm = host.default_tonemap_params()
    pos, nrm, mesh = _deform(s["mesh"], 5, amp=0.1)
    (_, ppos), (_, pnrm) = _pinned(pos), _pinned(nrm)
    want = []
    for m in (s["mesh"], mesh):
        r, _ = _fresh(w, h, ggx_lut, s, m, accel=False)
        with r:
            r.frame(cam.frame_params(tm))
            want.append(r.read_srgb8())
    assert want[0].tobytes() != want[1].tobytes()
    import torch
    a = torch.zeros(h * w * 4, dtype=torch.uint8).pin_memory().numpy().reshape(h, w, 4)
    with Renderer(w, h) as r:
        _upload_scene(r, ggx_lut, s)
        r.frame(cam.frame_params(tm))
        r.sync()
        r.frame(cam.frame_params(tm))
        r.read_srgb8_async(a)
        r.update_mesh_vertices(ppos, pnrm)
        r.frame(cam.frame_params(tm))
        r.wait_readback()
        b = r.read_srgb8()
    assert a.tobytes() == want[0].tobytes(), "frame A saw the new vertices"
    assert b.tobytes() == want[1].tobytes(), "frame B did not see the new vertices"


# ---------------------------------------------------------------------------------------------------------- 6. no blocking
def test_update_does_not_block(ggx_lut):
    """With the stream held up on the GPU, a page-locked update + the async top-level update + a frame return at once;
    tr_build_acceleration_structures in the same place waits for the GPU."""
    import torch
    w, h = 960, 540
    s = scenes.shadow_scene(w, h)
    fp = lambda hdl: s["camera"].frame_params(host.default_tonemap_params(), acceleration_structure_address=hdl)
    keep = [(_pinned(p), _pinned(n)) for p, n, _ in (_deform(s["mesh"], k) for k in range(3))]
    stream = torch.cuda.Stream(device=0)
    with Renderer(w, h) as r:
        r.set_stream(stream.cuda_stream)
        _upload_scene(r, ggx_lut, s)
        handle = r.build_acceleration_structures()
        for (_, p), (_, n) in keep[:2]:    # warm-up: chunk spheres, the builder's scratch, the frame buffers
            r.update_mesh_vertices(p, n)
            r.update_top_level_acceleration_structure_async()
            r.frame(fp(handle))
        r.sync()
        _hold(stream, 0.2)
        t0 = time.perf_counter()
        r.update_mesh_vertices(keep[2][0][1], keep[2][1][1])
        r.update_top_level_acceleration_structure_async()
        r.frame(fp(handle))
        enqueue = time.perf_counter() - t0
        r.sync()
        total = time.perf_counter() - t0
        _hold(stream, 0.2)
        t0 = time.perf_counter()
        r.build_acceleration_structures()
        blocking = time.perf_counter() - t0
        r.sync()
        r.set_stream(None)
    print(f"mesh update: enqueue {enqueue * 1e3:.1f} ms, frame done after {total * 1e3:.1f} ms; host build {blocking * 1e3:.1f} ms")
    assert total > 0.15, "the sleep did not hold up the stream"
    assert enqueue < 0.1, f"update + async top level + frame blocked for {enqueue * 1e3:.1f} ms"
    assert blocking > 0.15


# ---------------------------------------------------------------------------------------------------------- 7. group
def test_group_members_updated(ggx_lut):
    """3 members on one device, each updated before tr_group_frame: the frame equals one context's bit for bit."""
    w, h = 960, 540
    s = scenes.shadow_scene(w, h)
    cam = s["camera"]
    tm = host.default_tonemap_params()
    ranges = _vertex_ranges(s)
    a, b = ranges[0]
    pos, nrm, mesh = _deform(s["mesh"], 2, a, b, amp=0.1)
    r, handle = _fresh(w, h, ggx_lut, s, mesh)
    with r:
        r.frame(cam.frame_params(tm, acceleration_structure_address=handle))
        want = r.read_hdr(), r.read_srgb8()
    members = [Renderer(w, h) for _ in range(3)]
    try:
        for m in members:
            _upload_scene(m, ggx_lut, s)
            m.build_acceleration_structures()
        with RendererGroup(members) as g:
            g.frame(cam.frame_params(tm, acceleration_structure_address=1))
            for m in members:
                m.update_mesh_vertices(pos, nrm, first_vertex=a)
                m.update_top_level_acceleration_structure_async()
            g.frame(cam.frame_params(tm, acceleration_structure_address=1))   # each member's own handle goes in
            g.sync()
            got = g.read_hdr(), g.read_srgb8()
    finally:
        for m in members:
            m.close()
    assert got[0].tobytes() == want[0].tobytes(), "group HDR differs from one context"
    assert got[1].tobytes() == want[1].tobytes(), "group sRGB8 differs from one context"


# ---------------------------------------------------------------------------------------------------------- 8. rules
def test_rules(ggx_lut):
    w, h = 160, 90
    s = scenes.shadow_scene(w, h)
    cam = s["camera"]
    m = s["mesh"]
    nv = len(m["positions"])
    pos, nrm, mesh = _deform(m, 1)
    rng = np.random.default_rng(31)
    o, d, t = _random_rays(rng, 20000, [-8, 0, -10], [8, 6, 6])
    with Renderer(w, h) as r:
        with pytest.raises(TrError) as e:
            r.update_mesh_vertices(pos[:4], nrm[:4])                     # no mesh
        assert e.value.status == TR_ERR_STATE
        _upload_scene(r, ggx_lut, s)
        with pytest.raises(TrError) as e:
            r.update_mesh_vertices(pos[:4], nrm[:4], first_vertex=nv - 3)
        assert e.value.status == TR_ERR_INVALID_ARG
        with pytest.raises(TrError) as e:
            r.update_mesh_vertices(pos[:1], nrm[:1], first_vertex=nv)
        assert e.value.status == TR_ERR_INVALID_ARG
        from transmission_renderer_b200 import lib
        import ctypes as C
        assert lib().tr_update_mesh_vertices(r._ctx, C.c_uint32(0), C.c_uint32(4), None, None) == TR_ERR_INVALID_ARG
        r.frame(cam.frame_params())
        r.sync()
        before = Renderer.launch_count()
        r.update_mesh_vertices(pos[:0], nrm[:0], first_vertex=5)            # n = 0: nothing
        assert Renderer.launch_count() == before
        # an update before any build: the build picks it up
        r.update_mesh_vertices(pos, nrm)
        assert Renderer.launch_count() - before == MESH_UPDATE_LAUNCHES_NO_ACCEL
        handle = r.build_acceleration_structures()
        got = r.trace_shadow_rays(o, d, t)
        r.sync()
        before = Renderer.launch_count()
        r.update_mesh_vertices(pos, nrm)
        assert Renderer.launch_count() - before == MESH_UPDATE_LAUNCHES
        # a traced frame between the update and a top-level update is refused; after the update it runs
        with pytest.raises(TrError) as e:
            r.frame(cam.frame_params(acceleration_structure_address=handle))
        assert e.value.status == TR_ERR_STATE
        assert r.update_top_level_acceleration_structure_async() == handle
        r.frame(cam.frame_params(acceleration_structure_address=handle))
        # a new set_mesh: the call works on the new mesh
        r.set_mesh(m["positions"], m["normals"], m["uvs"], m["indices"])
        handle = r.build_acceleration_structures()
        r.update_mesh_vertices(pos, nrm)
        r.update_top_level_acceleration_structure()
        got2 = r.trace_shadow_rays(o, d, t)
        r.sync()
    fresh, _ = _fresh(w, h, ggx_lut, s, mesh)
    with fresh:
        want = fresh.trace_shadow_rays(o, d, t)
    assert np.array_equal(got, want) and np.array_equal(got2, want)
