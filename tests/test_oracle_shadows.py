"""Ray-queried shadows on the CPU oracle (oracle/shadow.c): known answers of trace_shadow_ray (shader/src/lighting.rs:97-125)
and of the top-level instance filter (src/main.rs:614-625), the tree walk against the tree-less definition, and the
effect on a shaded frame."""
import numpy as np
import pytest

from accel_checks import _surface_rays
from pipeline import oracle_cluster_lights, oracle_scene
from transmission_renderer_b200 import abi, host, scenes

f32 = np.float32


def _one_quad(bucket=0, translation=(0.0, 1.0, 0.0), scale=1.0, rotation=(0, 0, 0, 1)):
    meshes = scenes.MeshSet()
    q = meshes.add(scenes.quad_mesh(1.0), bucket)
    mesh, prims = meshes.arrays()
    inst = scenes.make_instance(translation, scale, rotation, q, 0)
    return mesh, prims, inst


def test_known_answers(oracle):
    mesh, prims, inst = _one_quad()                       # unit quad in the plane y = 1, x and z in [-1, 1]
    acc = oracle.Accel(mesh, inst, prims)
    assert acc.n_instances == 1
    up, down = (0.0, 1.0, 0.0), (0.0, -1.0, 0.0)
    cases = [
        ((0.0, 0.0, 0.0), up, 10.0, 0),                   # straight through the quad
        ((0.0, 2.0, 0.0), down, 10.0, 0),                 # both faces occlude (RayFlags::NONE, no culling)
        ((1.5, 0.0, 0.0), up, 10.0, 1),                   # passes beside it
        ((0.0, 0.0, 0.0), up, 0.9, 1),                    # t_max short of the hit (t = 1)
        ((0.0, 0.0, 0.0), up, 1.0, 1),                    # t < t_max is strict
        ((0.0, 0.0, 0.0), up, 1.0001, 0),
        ((0.0, 0.9995, 0.0), up, 10.0, 1),                # hit at t = 0.0005 < t_min = 0.001: no self-shadowing
        ((0.0, 0.998, 0.0), up, 10.0, 0),                 # t = 0.002 > t_min
        ((0.0, 0.0, 0.0), down, 10.0, 1),                 # pointing away
        ((0.3, 0.0, -0.2), (0.0, 0.6, 0.8), 10.0, 1),     # leaves through z > 1 before reaching y = 1 (t = 1.667 -> z = 1.13)
        ((0.3, 0.0, -0.2), (0.0, 0.8, 0.6), 10.0, 0),     # t = 1.25 -> z = 0.55: inside
    ]
    o, d, t, want = zip(*cases)
    got = acc.trace(np.array(o, f32), np.array(d, f32), np.array(t, f32))
    assert list(got) == list(want)
    assert list(acc.trace(np.array(o, f32), np.array(d, f32), np.array(t, f32), brute=True)) == list(want)


def test_instance_transform_and_top_level_filter(oracle):
    # the same quad, scaled by 3, lifted to y = 2 and rotated 90 degrees about z: it now stands in the plane x = 0
    rz = (0.0, 0.0, float(np.sin(np.pi / 4)), float(np.cos(np.pi / 4)))
    mesh, prims, inst = _one_quad(translation=(0.0, 2.0, 0.0), scale=3.0, rotation=rz)
    acc = oracle.Accel(mesh, inst, prims)
    o = np.array([(-5, 2, 0), (-5, 2, 2.9), (-5, 2, 3.1), (-5, 5.1, 0), (-5, -0.9, 0)], f32)
    d = np.tile(np.array([(1, 0, 0)], f32), (5, 1))
    assert list(acc.trace(o, d, np.full(5, 100.0, f32))) == [0, 0, 1, 1, 0]
    # t keeps its world meaning through the instance scale: the wall is 5 m away
    assert list(acc.trace(o[:1], d[:1], np.array([4.99], f32))) == [1] and list(acc.trace(o[:1], d[:1], np.array([5.01], f32))) == [0]
    # draw buffers 0 and 1 cast shadows, 2 and 3 (transmissive geometry) do not
    for bucket, casts in ((0, True), (1, True), (2, False), (3, False)):
        mesh, prims, inst = _one_quad(bucket=bucket)
        acc = oracle.Accel(mesh, inst, prims)
        assert acc.n_instances == (1 if casts else 0)
        lit = acc.trace(np.zeros((1, 3), f32), np.array([(0, 1, 0)], f32), np.array([10.0], f32))[0]
        assert lit == (0 if casts else 1)


def test_tree_walk_equals_the_definition(oracle):
    """The hierarchy only skips work: its answer is the tree-less definition's answer for every ray."""
    s = scenes.shadow_scene(320, 180)
    acc = oracle.Accel(s["mesh"], s["instances"], s["primitives"])
    assert acc.n_instances == 7                                         # everything but the glass knot
    rng = np.random.default_rng(5)
    n = 30000
    o = rng.uniform([-8, 0, -10], [8, 6, 6], (n, 3)).astype(f32)
    d = rng.normal(size=(n, 3))
    d = (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(f32)
    d[::7, rng.integers(0, 3)] = 0.0                                    # axis-parallel components: the 0 * inf corner of the slab test
    d[::11] = np.sign(d[::11]) * (np.abs(d[::11]) > 0.5)                # exactly axis-aligned / diagonal, some components -0
    t = rng.uniform(0.5, 40, n).astype(f32)
    ok = np.linalg.norm(d, axis=1) > 0
    o, d, t = o[ok], d[ok], t[ok]
    a, b = acc.trace(o, d, t), acc.trace(o, d, t, brute=True)
    assert (a != b).sum() == 0
    assert 0.05 < 1 - a.mean() < 0.95
    po, pd, pt = _surface_rays(s, oracle, 20000, rng)
    a, b = acc.trace(po, pd, pt), acc.trace(po, pd, pt, brute=True)
    assert (a != b).sum() == 0 and 0.05 < 1 - a.mean() < 0.95


def test_shadows_darken_the_frame(oracle, ggx_lut):
    w, h = 160, 90
    s = scenes.shadow_scene(w, h)
    cam = s["camera"]
    pc = cam.push_constants()
    _, visible = oracle.frustum_culling(s["instances"], s["primitives"], cam.culling())
    g0, g1 = oracle.visibility(s["mesh"], s["instances"], s["primitives"], visible, pc)
    _, cc, ci = oracle_cluster_lights(oracle, cam, s["uniforms"], s["lights"])
    sc = oracle_scene(pc, s["uniforms"], s["materials"], s["lights"], cc, ci)
    lit32, _ = oracle.shade_opaque_frame(g0, sc)
    sc["accel"] = oracle.Accel(s["mesh"], s["instances"], s["primitives"])
    sh32, sh16 = oracle.shade_opaque_frame(g0, sc)
    assert (sh32[..., :3] <= lit32[..., :3] * (1 + 1e-6) + 1e-7).all()          # a shadow factor never adds light
    darker = (sh32[..., :3].sum(-1) < 0.8 * lit32[..., :3].sum(-1)) & (g0["depth"] > 0)
    assert 0.02 < darker.mean() < 0.9
    mask = oracle.shadow_mask_frame(g0, sc)
    covered = g0["depth"] > 0
    assert mask[:, ~covered].sum() == 0 and (mask[4][covered] & 1).mean() > 0.02      # the sun is blocked somewhere
    # a fully lit pixel (no occluded ray) is shaded exactly as without ray queries
    none = covered & (mask.sum(0) == 0)
    assert none.sum() > 100 and np.array_equal(sh32[none], lit32[none])
    # the glass receives shadows too (lighting.rs:25-35, 64-75)
    levels = oracle.build_pyramid(sh16)
    t32, _ = oracle.shade_transmission_frame(g1, sc, levels, ggx_lut, sh32, sh16)
    sc_lit = dict(sc, accel=None)
    t32_lit, _ = oracle.shade_transmission_frame(g1, sc_lit, levels, ggx_lut, sh32, sh16)
    glass = g1["depth"] > 0
    assert glass.sum() > 50 and (np.abs(t32[glass] - t32_lit[glass]).max() > 1e-3)


def test_slab_is_monotone_in_the_box(oracle):
    """What makes the result independent of the trees: a box that contains another one never fails where the inner one
    passes — including rays with zero and negative-zero direction components and origins on a face (0 * inf)."""
    from hypothesis import given, settings, strategies as st
    coord = st.one_of(st.floats(-50, 50, width=32), st.sampled_from([0.0, 1.0, -1.0, 0.5]))
    comp = st.one_of(st.floats(-1, 1, width=32), st.sampled_from([0.0, -0.0, 1.0, -1.0]))
    grow = st.one_of(st.floats(0, 10, width=32), st.just(0.0))

    @settings(max_examples=1500, deadline=None)
    @given(st.tuples(coord, coord, coord), st.tuples(comp, comp, comp), st.tuples(coord, coord, coord), st.tuples(grow, grow, grow),
           st.tuples(grow, grow, grow), st.tuples(grow, grow, grow), st.floats(0.015625, 100, width=32))
    def check(o, d, lo, ext, g_lo, g_hi, t_max):
        if d == (0.0, 0.0, 0.0):
            return
        lo = np.array(lo, f32)
        hi = (lo + np.array(ext, f32)).astype(f32)
        big_lo = (lo - np.array(g_lo, f32)).astype(f32)
        big_hi = (hi + np.array(g_hi, f32)).astype(f32)
        if oracle.slab_test(o, d, 0.001, t_max, lo, hi):
            assert oracle.slab_test(o, d, 0.001, t_max, big_lo, big_hi)

    check()
    # known answers of the 0 * inf corner: direction parallel to a face the origin lies on
    assert oracle.slab_test((0, 0, 0), (1, 0, 0), 0.001, 10, (1, 0, -1), (2, 1, 1))          # origin.y == lo.y, d.y == 0
    assert not oracle.slab_test((0, -0.5, 0), (1, 0, 0), 0.001, 10, (1, 0, -1), (2, 1, 1))   # below the box, parallel
    assert oracle.slab_test((0, 0.5, 0), (1, -0.0, 0), 0.001, 10, (1, 0, -1), (2, 1, 1))     # negative zero component
