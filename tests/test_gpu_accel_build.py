"""tr_build_acceleration_structures_async: the bottom level built on the device in stream order (H-PLOC, single-triangle
leaves), then the top level.  The trees differ from the host's binned-SAH trees; the occlusion result is defined without the
trees (DESIGN.md section 7 N4), so a context built with the async call must trace and render exactly what a context built
with the blocking call traces and renders on the same arrays, and both must match the brute-force definition."""
import time

import numpy as np
import pytest

from accel_checks import ACCEL_STACK, ASYNC_TLAS_LAUNCHES
from accel_checks import _check_blas, _deform, _hold, _pinned, _random_rays, _records_key, _reference, _surface_rays, _tree_checks, _upload_scene
from pipeline import REL_L2_TOL, rel_l2
from transmission_renderer_b200 import Renderer, RendererGroup, TrError, abi, host, scenes

pytestmark = pytest.mark.gpu
f32 = np.float32
TR_ERR_INVALID_ARG, TR_ERR_STATE = -1, -6


def _async_build_launches(n_prims):
    """async_blas_launches (k_accel_build.cu) + the top level: counts, 2 scans, init, bounds, codes, 5 per radix pass,
    H-PLOC, placement, reset, H-PLOC, placement; ceil((30 + bits of the largest primitive id) / 8) radix passes."""
    bits = int(n_prims - 1).bit_length()
    return 11 + 5 * ((30 + bits + 7) // 8) + ASYNC_TLAS_LAUNCHES


# ---------------------------------------------------------------------------------------------------------- scenes
def _knot_scene(w, h, n_u=768, n_v=64):
    """The shadow scene plus a large torus knot (one primitive, two instances) above the ground."""
    s = scenes.shadow_scene(w, h)
    pos, nrm, uv, idx = scenes.torus_knot(n_u=n_u, n_v=n_v)
    return _with_primitives(s, [(pos, nrm, uv, idx, 0)], [((0.0, 2.5, -2.0), 2.0, 0), ((3.0, 1.5, -4.0), 1.2, 0)])


def _with_primitives(s, extra, placements):
    """Scene s plus primitives extra = [(positions, normals, uvs, indices, draw_buffer_index)] and instances placements =
    [(translation, scale, index into extra)]."""
    m = s["mesh"]
    pos, nrm, uv, idx = [m["positions"]], [m["normals"]], [m["uvs"]], [m["indices"]]
    v0, i0 = len(m["positions"]), len(m["indices"])
    prims = []
    for p_pos, p_nrm, p_uv, p_idx, bucket in extra:
        p = np.zeros(1, abi.primitive_info)
        with np.errstate(all="ignore"):
            fin = p_pos[np.isfinite(p_pos).all(1)] if len(p_pos) else np.zeros((1, 3), f32)
            fin = fin if len(fin) else np.zeros((1, 3), f32)
            lo, hi = fin.min(0).astype(np.float64), fin.max(0).astype(np.float64)
        p["packed_bounding_sphere"][0] = (*((lo + hi) / 2), np.linalg.norm(hi - lo) / 2 + 1.0)
        p["index_count"] = len(p_idx)
        p["first_index"] = i0
        p["draw_buffer_index"] = bucket
        prims.append(p)
        pos.append(p_pos.astype(f32)); nrm.append(p_nrm.astype(f32)); uv.append(p_uv.astype(f32))
        idx.append(p_idx.astype(np.uint32) + np.uint32(v0))
        v0 += len(p_pos)
        i0 += len(p_idx)
    first = len(s["primitives"])
    inst = [scenes.make_instance(t, sc, (0.0, 0.0, 0.0, 1.0), first + k, 0) for t, sc, k in placements]
    mesh = dict(positions=np.concatenate(pos), normals=np.concatenate(nrm), uvs=np.concatenate(uv), indices=np.concatenate(idx))
    return dict(s, mesh=mesh, primitives=np.concatenate([s["primitives"]] + prims), instances=np.concatenate([s["instances"]] + inst))


def _soup(tri_pos):
    """A triangle soup (n, 3, 3) as (positions, normals, uvs, indices)."""
    p = np.ascontiguousarray(tri_pos, f32).reshape(-1, 3)
    n = np.tile(np.array([0.0, 1.0, 0.0], f32), (len(p), 1))
    return p, n, np.zeros((len(p), 2), f32), np.arange(len(p), dtype=np.uint32)


def _scene(kind, w, h):
    if kind == "shadow":
        return scenes.shadow_scene(w, h), ([-8, 0, -10], [8, 6, 6])
    if kind == "instanced":
        return scenes.instanced_scene(w, h, n_instances=2000, n_lights=16), ([-30, 0, -30], [30, 12, 30])
    return _knot_scene(w, h), ([-8, 0, -10], [8, 6, 6])


# ---------------------------------------------------------------------------------------------------------- structure
def _predicted(prims):
    nt = prims["index_count"].astype(np.int64) // 3
    sizes = np.maximum(1, nt - 1)
    return np.concatenate([[0], np.cumsum(sizes)[:-1]]), np.concatenate([[0], np.cumsum(nt)[:-1]]), int(sizes.sum()), nt


def _area(lo, hi):
    d = (hi - lo).astype(np.float64)
    return d[..., 0] * d[..., 1] + d[..., 1] * d[..., 2] + d[..., 2] * d[..., 0]


def _trees(nodes, prims, roots=None):
    """Per primitive (root, end, depth, SAH cost); the trees lie one after the other, each root first."""
    out = []
    if roots is None:   # the host build: count each tree's nodes
        roots, r = [], 0
        for p in range(len(prims)):
            roots.append(r)
            todo, n = [r], 0
            while todo:
                k = todo.pop()
                n += 1
                todo += [c for c in (int(nodes["c0"][k]), int(nodes["c1"][k])) if c >= 0]
            r += n
    for p, root in enumerate(roots):
        end = roots[p + 1] if p + 1 < len(roots) else len(nodes)
        sub = nodes[root:end]
        depth, todo = 0, [(root, 1)]
        while todo:
            k, d = todo.pop()
            depth = max(depth, d)
            for c in (int(nodes["c0"][k]), int(nodes["c1"][k])):
                if c >= 0:
                    assert root < c < end and c > k, f"primitive {p}: node {k} -> {c} leaves its tree or precedes its parent"
                    todo.append((c, d + 1))
        cost = None
        if end - root > 1 or sub["c0"][0] != sub["c1"][0]:
            lo = np.minimum(sub["lo0"], sub["lo1"])
            hi = np.maximum(sub["hi0"], sub["hi1"])
            cost = float(_area(lo, hi).sum())
            for side in ("0", "1"):
                c = sub["c" + side].astype(np.int64)
                leaf = c < 0
                count = ((~c[leaf] & 0xFFFFFFFF) >> 28) + 1
                cost += float((_area(sub["lo" + side][leaf], sub["hi" + side][leaf]) * count).sum())
            root_area = _area(lo[0], hi[0])
            cost = cost / root_area if root_area > 0 else None
        out.append((root, end, depth, cost))
    return out


def _check_device_tree(nodes, tris, prims, mesh):
    """Layout, leaves and boxes of an async build; returns the per-primitive (root, end, depth, cost)."""
    roots, bases, total, nt = _predicted(prims)
    assert len(nodes) == total, "node count is not sum max(1, nt - 1)"
    assert len(tris) == int(nt.sum())
    assert (nodes["pad"] == 0).all()
    trees = _trees(nodes, prims, list(roots))
    for p, (root, end, depth, _) in enumerate(trees):
        assert depth < ACCEL_STACK, f"primitive {p}: depth {depth}"
        sub = nodes[root:end]
        refs = np.concatenate([sub["c0"], sub["c1"]]).astype(np.int64)
        leaves = np.sort(~refs[refs < 0] & 0xFFFFFFFF)
        if nt[p] >= 2:   # single-triangle leaves: every triangle of the primitive exactly once
            assert np.array_equal(leaves, np.arange(nt[p])), f"primitive {p}: leaves are not 0..{nt[p] - 1} once each"
    if not np.isnan(mesh["positions"]).any():   # the restatement's min / max would keep a NaN that fminf / fmaxf drop
        _check_blas(nodes, tris, prims, mesh)   # per primitive: the mesh's triangles as a multiset; exact-union boxes
    return trees


def _build_pair(lut, s, w=160, h=90):
    """(host context, async context) on the same arrays, with their handles."""
    rh, ra = Renderer(w, h), Renderer(w, h)
    _upload_scene(rh, lut, s)
    _upload_scene(ra, lut, s)
    return rh, rh.build_acceleration_structures(), ra, ra.build_acceleration_structures_async()


# ---------------------------------------------------------------------------------------------------------- 1-2, 5. rays, structure, quality
@pytest.mark.parametrize("kind", ["shadow", "instanced", "knot"])
def test_rays_structure_quality(oracle, ggx_lut, kind):
    w, h = 320, 180
    s, box = _scene(kind, w, h)
    rng = np.random.default_rng(41)
    o, d, t = _random_rays(rng, 200000, *box)
    po, pd, pt = _surface_rays(s, oracle, 100000, rng)
    rh, hh, ra, ha = _build_pair(ggx_lut, s, w, h)
    with rh, ra:
        assert ha == ra.update_top_level_acceleration_structure_async()
        want = rh.trace_shadow_rays(o, d, t), rh.trace_shadow_rays(po, pd, pt)
        got = ra.trace_shadow_rays(o, d, t), ra.trace_shadow_rays(po, pd, pt)
        hn, _ = rh.read_bottom_level_acceleration_structure()
        an, at = ra.read_bottom_level_acceleration_structure()
        _, hi = rh.read_top_level_acceleration_structure()
        tn, ai = ra.read_top_level_acceleration_structure()
    for g, wnt in zip(got, want):
        assert (g != wnt).sum() == 0, f"{(g != wnt).sum()} rays differ from the host-built context"
    assert 0.02 < 1 - want[0].mean() < 0.98
    acc = oracle.Accel(s["mesh"], s["instances"], s["primitives"])
    sub = slice(0, 20000)
    assert np.array_equal(got[0][sub], acc.trace(o[sub], d[sub], t[sub], brute=True))
    assert np.array_equal(got[1][sub], acc.trace(po[sub], pd[sub], pt[sub], brute=True))
    prims = s["primitives"]
    trees = _check_device_tree(an, at, prims, s["mesh"])
    # the top level: the host's records (boxes from the per-primitive table) apart from the roots, which are the predicted ones
    roots = set(int(r) for r in _predicted(prims)[0])
    assert set(int(r) for r in ai["blas_root"]) <= roots
    assert _records_key(ai).tobytes() == _records_key(hi).tobytes(), "top-level records differ from the host build's"
    assert _tree_checks(tn, ai) < ACCEL_STACK
    # quality: SAH cost against the host tree, primitive by primitive
    host_trees = _trees(hn, prims)
    nt = prims["index_count"] // 3
    ratios = [(a[3] / b[3], int(nt[p])) for p, (a, b) in enumerate(zip(trees, host_trees))
              if nt[p] >= 16 and a[3] is not None and b[3] is not None]
    depth = max(tr[2] for tr in trees)
    print(f"{kind}: SAH cost device / host per primitive (triangles): "
          + ", ".join(f"{r:.3f} ({n})" for r, n in sorted(ratios, key=lambda x: -x[1])[:8])
          + f"; max {max(r for r, _ in ratios):.3f}; max depth {depth}")
    assert max(r for r, _ in ratios) <= 1.2


# ---------------------------------------------------------------------------------------------------------- 2. nt = 0 / 1 roots, 4. pathological
def _pathological(case):
    rng = np.random.default_rng(7)
    if case == "equal_centroids":     # 4096 triangles around one centroid
        a = rng.normal(size=(4096, 3)) * 0.5
        tri = np.stack([a, -a, np.zeros_like(a)], 1)
        return [(_soup(tri), 0)]
    if case == "geometric_chain":     # sizes 2^-k, k = 0..199, each in the corner of the previous
        k = np.arange(200)
        sc = 2.0 ** -k.astype(np.float64)
        base = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0.5]], np.float64)
        tri = base[None] * sc[:, None, None] + np.array([0.1, 0.2, 0.0])
        return [(_soup(tri), 0)]
    if case == "ten_decades":         # scales 1e-5 .. 1e5, and a primitive near 1e30
        sc = 10.0 ** rng.uniform(-5, 5, 3000)
        c = rng.normal(size=(3000, 3)) * 3
        tri = c[:, None] + rng.normal(size=(3000, 3, 3)) * sc[:, None, None]
        far = rng.normal(size=(500, 3, 3)) * 1e29 + 1e30
        return [(_soup(tri), 0), (_soup(far), 0)]
    if case == "degenerate_nonfinite":
        tri = rng.normal(size=(2000, 3, 3)) * 2
        tri[::5, 1] = tri[::5, 0]                     # two equal vertices
        tri[1::5, :] = tri[1::5, :1]                  # a point
        tri[2::17, 0, 0] = np.nan
        tri[3::19, 1, 1] = np.inf
        tri[4::23, 2, 2] = -np.inf
        tri[5::29, :, :] = np.nan                     # every vertex NaN
        return [(_soup(tri), 0)]
    if case == "tiny_next_to_huge":   # primitives of 0-3 triangles around one of more than 2^20
        pos, nrm, uv, idx = scenes.torus_knot(n_u=4200, n_v=128)
        small = [_soup(rng.normal(size=(n, 3, 3))) for n in (0, 1, 2, 3)]
        return [(small[0], 0), (small[1], 0), ((pos, nrm, uv, idx), 0), (small[2], 1), (small[3], 0), (small[1], 2)]
    raise ValueError(case)


@pytest.mark.parametrize("case", ["equal_centroids", "geometric_chain", "ten_decades", "degenerate_nonfinite", "tiny_next_to_huge",
                                  "forced_fallback"])
def test_pathological_inputs(oracle, ggx_lut, monkeypatch, case):
    w, h = 160, 90
    base = scenes.shadow_scene(w, h)
    if case == "forced_fallback":     # every primitive rebuilt as the radix tree
        monkeypatch.setenv("TR_ACCEL_DEPTH_LIMIT", "0")
        s = _knot_scene(w, h, n_u=256, n_v=32)
    else:
        extra = _pathological(case)
        placements = [((0.5 * k, 1.0, -2.0 - k), 1.0, k) for k in range(len(extra))]
        s = _with_primitives(base, [(*g, b) for g, b in extra], placements)
    rng = np.random.default_rng(43)
    o, d, t = _random_rays(rng, 100000, [-8, -1, -10], [8, 6, 6])
    huge = case == "tiny_next_to_huge"
    rh, hh, ra, ha = _build_pair(ggx_lut, s, w, h)
    with rh, ra:
        want = rh.trace_shadow_rays(o, d, t)
        got = ra.trace_shadow_rays(o, d, t)
        hn, ht = rh.read_bottom_level_acceleration_structure()
        an, at = ra.read_bottom_level_acceleration_structure()
    assert (got != want).sum() == 0, f"{(got != want).sum()} rays differ from the host-built context"
    prims = s["primitives"]
    trees = _check_device_tree(an, at, prims, s["mesh"])
    print(f"{case}: max depth {max(tr[2] for tr in trees)}")
    # the nt = 0 and nt = 1 trees are the host's, byte for byte
    roots, bases, _, nt = _predicted(prims)
    host_trees = _trees(hn, prims)
    for p in np.nonzero(nt <= 1)[0]:
        hr = host_trees[p][0]
        assert an[roots[p]].tobytes() == hn[hr].tobytes(), f"primitive {p} ({nt[p]} triangles)"
        if nt[p] == 1:
            assert at[bases[p]].tobytes() == ht[bases[p]].tobytes()
    sub = slice(0, 300 if huge else 5000)
    acc = oracle.Accel(s["mesh"], s["instances"], s["primitives"])
    assert np.array_equal(got[sub], acc.trace(o[sub], d[sub], t[sub], brute=True))


# ---------------------------------------------------------------------------------------------------------- 3. determinism
def test_deterministic(ggx_lut):
    w, h = 160, 90
    s = _knot_scene(w, h)
    out = []
    with Renderer(w, h) as a, Renderer(w, h) as b:
        _upload_scene(a, ggx_lut, s)
        _upload_scene(b, ggx_lut, s)
        for r in (a, a, b):
            r.build_acceleration_structures_async()
            out.append(r.read_bottom_level_acceleration_structure() + r.read_top_level_acceleration_structure())
    for k in (1, 2):
        for x, y in zip(out[0], out[k]):
            assert x.tobytes() == y.tobytes(), f"build {k} differs from build 0"


# ---------------------------------------------------------------------------------------------------------- 6. frames
def test_frames_match_host_build(ggx_lut):
    w, h = 480, 270
    s = _knot_scene(w, h)
    cam = s["camera"]
    tm = host.default_tonemap_params()
    res = []
    for mode in ("host", "async", "async+host_tlas", "async+async_tlas"):
        with Renderer(w, h) as r:
            _upload_scene(r, ggx_lut, s)
            handle = r.build_acceleration_structures() if mode == "host" else r.build_acceleration_structures_async()
            if mode.endswith("host_tlas"):
                r.set_instances(s["instances"])
                assert r.update_top_level_acceleration_structure() == handle
            elif mode.endswith("async_tlas"):
                r.set_instances(s["instances"])
                assert r.update_top_level_acceleration_structure_async() == handle
            r.frame(cam.frame_params(tm, acceleration_structure_address=handle))
            res.append((r.read_shadow_mask(0), r.read_shadow_mask(1), r.read_hdr(), r.read_srgb8()))
    assert (res[0][0] == 0).any() and (res[0][0] != 0).any()
    for k in range(1, len(res)):
        for name, a, b in zip(("opaque mask", "transmissive mask", "HDR", "sRGB8"), res[k], res[0]):
            assert a.tobytes() == b.tobytes(), f"mode {k}: {name} differs"


def test_animation_refit_and_rebuild(oracle, ggx_lut):
    """8 deformed frames: refit every frame, async rebuild every third; each frame equals a fresh context's (blocking build),
    the last one the oracle's."""
    w, h = 480, 270
    s = scenes.shadow_scene(w, h)
    cam = s["camera"]
    tm = host.default_tonemap_params()
    meshes = []
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
            handle = r.build_acceleration_structures_async()
            for k, ((_, pos), (_, nrm), m) in enumerate(meshes):
                r.update_mesh_vertices(pos, nrm)
                if k % 3 == 2:
                    assert r.build_acceleration_structures_async() == handle
                    nodes, tris = r.read_bottom_level_acceleration_structure()
                    _check_device_tree(nodes, tris, s["primitives"], m)
                else:
                    assert r.update_top_level_acceleration_structure_async() == handle
                    if k == 1:   # the refit of an async-built tree: same topology, exact unions
                        nodes, tris = r.read_bottom_level_acceleration_structure()
                        _check_blas(nodes, tris, s["primitives"], m)
                r.frame(cam.frame_params(tm, acceleration_structure_address=handle))
                got = outputs(r)
                fresh.set_mesh(m["positions"], m["normals"], m["uvs"], m["indices"])
                fresh.frame(cam.frame_params(tm, acceleration_structure_address=fresh.build_acceleration_structures()))
                want = outputs(fresh)
                for name, a, b in zip(("opaque mask", "transmissive mask", "HDR", "sRGB8"), got, want):
                    assert a.tobytes() == b.tobytes(), f"frame {k}: {name} differs"
            last32 = r.read_hdr_f32()
    finally:
        fresh.close()
    s2 = dict(s, mesh=meshes[-1][2])
    ref = _reference(oracle, ggx_lut, s2, oracle.Accel(s2["mesh"], s2["instances"], s2["primitives"]))
    assert (got[0] != oracle.shadow_mask_frame(ref["g0"], ref["scene"])).sum() == 0
    assert (got[1] != oracle.shadow_mask_frame(ref["g1"], ref["scene"])).sum() == 0
    assert rel_l2(last32[..., :3], ref["t32"][..., :3]) < REL_L2_TOL


# ---------------------------------------------------------------------------------------------------------- 7. rules
def test_does_not_block(ggx_lut):
    """With the stream held up on the GPU, the async build after a tr_set_mesh + a frame return at once, alone and on the
    members of a 3-context group; the blocking build in the same place waits.  tr_set_mesh (pageable arrays) is enqueued
    before the stream is held: the build reads the new mesh in stream order."""
    import torch
    w, h = 960, 540
    s = _knot_scene(w, h)
    m = s["mesh"]
    fp = lambda hdl: s["camera"].frame_params(host.default_tonemap_params(), acceleration_structure_address=hdl)
    stream = torch.cuda.Stream(device=0)
    with Renderer(w, h) as r:
        r.set_stream(stream.cuda_stream)
        _upload_scene(r, ggx_lut, s)
        for _ in range(2):   # warm-up: buffers and scratch
            r.frame(fp(r.build_acceleration_structures_async()))
        r.sync()
        r.set_mesh(m["positions"], m["normals"], m["uvs"], m["indices"])
        _hold(stream, 0.2)
        t0 = time.perf_counter()
        r.frame(fp(r.build_acceleration_structures_async()))
        enqueue = time.perf_counter() - t0
        r.sync()
        total = time.perf_counter() - t0
        _hold(stream, 0.2)
        t0 = time.perf_counter()
        r.build_acceleration_structures()
        blocking = time.perf_counter() - t0
        r.sync()
        r.set_stream(None)
    print(f"async build: enqueue {enqueue * 1e3:.1f} ms, frame done after {total * 1e3:.1f} ms; host build {blocking * 1e3:.1f} ms")
    assert total > 0.15, "the sleep did not hold up the stream"
    assert enqueue < 0.1, f"async build + frame blocked for {enqueue * 1e3:.1f} ms"
    assert blocking > 0.15

    cam = s["camera"]
    tm = host.default_tonemap_params()
    with Renderer(w, h) as r:
        _upload_scene(r, ggx_lut, s)
        r.frame(cam.frame_params(tm, acceleration_structure_address=r.build_acceleration_structures()))
        want = r.read_hdr(), r.read_srgb8()
    members = [Renderer(w, h) for _ in range(3)]
    try:
        members[0].set_stream(stream.cuda_stream)
        for r in members:
            _upload_scene(r, ggx_lut, s)
        with RendererGroup(members) as g:
            for _ in range(2):
                for r in members:
                    r.build_acceleration_structures_async()
                g.frame(cam.frame_params(tm, acceleration_structure_address=1))
            g.sync()
            for r in members:
                r.set_mesh(m["positions"], m["normals"], m["uvs"], m["indices"])
            _hold(stream, 0.2)
            t0 = time.perf_counter()
            for r in members:
                r.build_acceleration_structures_async()
            g.frame(cam.frame_params(tm, acceleration_structure_address=1))
            enqueue = time.perf_counter() - t0
            g.sync()
            total = time.perf_counter() - t0
            got = g.read_hdr(), g.read_srgb8()
        members[0].set_stream(None)
    finally:
        for r in members:
            r.close()
    print(f"group: enqueue {enqueue * 1e3:.1f} ms, frame done after {total * 1e3:.1f} ms")
    assert got[0].tobytes() == want[0].tobytes() and got[1].tobytes() == want[1].tobytes()
    assert total > 0.15 and enqueue < 0.1


def test_rules(ggx_lut):
    w, h = 160, 90
    s = scenes.shadow_scene(w, h)
    cam = s["camera"]
    m = s["mesh"]
    with Renderer(w, h) as r:
        with pytest.raises(TrError) as e:
            r.build_acceleration_structures_async()                               # nothing bound
        assert e.value.status == TR_ERR_STATE
        _upload_scene(r, ggx_lut, s)
        handle = r.build_acceleration_structures()
        assert r.build_acceleration_structures_async() == handle                 # same handle as the blocking call
        r.sync()
        before = Renderer.launch_count()
        assert r.build_acceleration_structures_async() == handle
        assert Renderer.launch_count() - before == _async_build_launches(len(s["primitives"]))
        r.frame(cam.frame_params(acceleration_structure_address=handle))
        # tr_set_mesh and tr_set_primitives invalidate the structures
        r.set_mesh(m["positions"], m["normals"], m["uvs"], m["indices"])
        with pytest.raises(TrError) as e:      # the handle is refused until the next build, as after the blocking one
            r.frame(cam.frame_params(acceleration_structure_address=handle))
        assert e.value.status == TR_ERR_INVALID_ARG and "acceleration_structure_address" in str(e.value)
        assert r.build_acceleration_structures_async() == handle
        r.frame(cam.frame_params(acceleration_structure_address=handle))
        r.set_primitives(s["primitives"])
        with pytest.raises(TrError) as e:
            r.frame(cam.frame_params(acceleration_structure_address=handle))
        assert e.value.status == TR_ERR_INVALID_ARG and "acceleration_structure_address" in str(e.value)
        assert r.build_acceleration_structures_async() == handle
        # a primitive past the index buffer, an instance naming a missing primitive: refused before anything is enqueued
        bad = s["primitives"].copy()
        bad["index_count"][1] = len(m["indices"])
        r.set_primitives(bad)
        r.sync()
        before = Renderer.launch_count()
        with pytest.raises(TrError) as e:
            r.build_acceleration_structures_async()
        assert e.value.status == TR_ERR_INVALID_ARG and "primitive 1" in str(e.value)
        assert Renderer.launch_count() == before
        r.set_primitives(s["primitives"])
        inst = s["instances"].copy()
        inst["primitive_id"][3] = 99
        r.set_instances(inst)
        with pytest.raises(TrError) as e:
            r.build_acceleration_structures_async()
        assert e.value.status == TR_ERR_INVALID_ARG and "instance 3" in str(e.value)
        r.set_instances(s["instances"])
        assert r.build_acceleration_structures_async() == handle
        r.frame(cam.frame_params(acceleration_structure_address=handle))
        r.sync()
    with Renderer(w, h) as r:
        _upload_scene(r, ggx_lut, s)
        r.set_primitives(s["primitives"][:0])
        with pytest.raises(TrError) as e:
            r.build_acceleration_structures_async()                               # no primitives
        assert e.value.status == TR_ERR_STATE
