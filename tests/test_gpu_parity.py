"""GPU parity tests: libtr.so (through the C ABI) against the CPU oracle on the same inputs.

Tolerances (BASELINE.json north_star): relative L2 <= 1e-4 on linear HDR, <= 2/255 per sRGB8
channel; every integer / index / fp16-bit-pattern result of the discrete stages bit-exact.
"""
import numpy as np
import pytest

from pipeline import REL_L2_TOL, SRGB_TOL, gpu_setup, oracle_cluster_lights, oracle_scene, rel_l2
from transmission_renderer_b200 import Renderer, abi, host, scenes

pytestmark = pytest.mark.gpu
f32 = np.float32


def _rand_unit(rng, n):
    v = rng.standard_normal((n, 3))
    return v / np.linalg.norm(v, axis=1, keepdims=True)


def _hemisphere(rng, n, normal, margin=0.0):
    v = _rand_unit(rng, n)
    s = np.sign(np.sum(v * normal, axis=1, keepdims=True))
    v = v * np.where(s == 0, 1, s) + margin * normal
    return v / np.linalg.norm(v, axis=1, keepdims=True)


def _rand_materials(rng, n, rough_lo=0.05):
    m = np.zeros(n, dtype=abi.material_params)
    m["diffuse_colour"] = rng.uniform(0.05, 1.0, (n, 3))
    m["metallic"] = rng.choice([0.0, 1.0, 0.3], n)
    m["perceptual_roughness"] = rng.uniform(rough_lo, 1.0, n)
    m["index_of_refraction"] = rng.uniform(1.0, 2.2, n)
    m["specular_colour"] = rng.uniform(0.2, 1.0, (n, 3))
    m["specular_factor"] = rng.uniform(0.0, 1.0, n)
    return m


# ------------------------------------------------------------------------------ glam-pbr contracts
def test_eval_basic_brdf(oracle):
    rng = np.random.default_rng(100)
    n = 200000
    p = np.zeros(n, dtype=abi.basic_brdf_params)
    nrm = _rand_unit(rng, n).astype(f32)
    p["normal"] = nrm
    # contract: shading vectors are normalised (glam-pbr lib.rs:47); normalise in f32 like a caller would
    for k in ("view", "light"):
        v = _hemisphere(rng, n, nrm).astype(f32)
        p[k] = v / np.linalg.norm(v, axis=1, keepdims=True).astype(f32)
    p["light_intensity"] = rng.uniform(0.1, 20.0, (n, 3))
    p["material_params"] = _rand_materials(rng, n)
    with Renderer(64, 64) as r:
        got = r.eval_basic_brdf(p)
    ref = oracle.eval_basic_brdf(p)
    assert rel_l2(got["diffuse"], ref["diffuse"]) < 2e-6
    assert rel_l2(got["specular"], ref["specular"]) < 2e-6   # the n.h chain is reproduced exactly
    np.testing.assert_allclose(got["specular"], ref["specular"], rtol=2e-5, atol=1e-7)
    np.testing.assert_allclose(got["diffuse"], ref["diffuse"], rtol=2e-5, atol=1e-7)


def test_eval_transmission_btdf(oracle):
    rng = np.random.default_rng(101)
    n = 200000
    p = np.zeros(n, dtype=abi.transmission_btdf_params)
    nrm = _rand_unit(rng, n).astype(f32)
    p["normal"] = nrm
    p["view"] = _hemisphere(rng, n, nrm).astype(f32)
    p["light"] = _rand_unit(rng, n).astype(f32)
    p["material_params"] = _rand_materials(rng, n)
    with Renderer(64, 64) as r:
        got = r.eval_transmission_btdf(p)
    ref = oracle.eval_transmission_btdf(p)
    assert rel_l2(got, ref) < 2e-6
    ok = np.isfinite(ref).all(axis=1)
    np.testing.assert_allclose(got[ok], ref[ok], rtol=3e-5, atol=1e-7)


def test_eval_ibl_volume_refraction(oracle, ggx_lut):
    rng = np.random.default_rng(102)
    w, h = 256, 128
    mip0 = np.ones((h, w, 4), dtype=f32)
    mip0[..., :3] = rng.uniform(0, 4, (h, w, 3)) * (rng.random((h, w, 1)) > 0.5)
    bits = oracle.f16_bits(mip0)
    levels = oracle.build_pyramid(bits)
    view = host.look_at_rh((0, 1, 4), (0, 0, 0), (0, 1, 0))
    pv = (host.perspective_matrix_reversed(w, h) @ view).astype(f32)
    n = 50000
    p = np.zeros(n, dtype=abi.ibl_volume_refraction_params)
    p["material_params"] = _rand_materials(rng, n)
    p["material_params"]["index_of_refraction"] = rng.uniform(1.05, 2.0, n)
    p["framebuffer_size_x"] = w
    nrm = _rand_unit(rng, n).astype(f32)
    p["position"] = rng.uniform(-1.5, 1.5, (n, 3))
    p["normal"] = nrm
    p["view"] = _hemisphere(rng, n, nrm, 0.1).astype(f32)
    p["thickness"] = rng.uniform(0, 1, n)
    p["model_scale"] = rng.uniform(0.5, 2, n)
    p["attenuation_distance"] = np.where(rng.random(n) < 0.3, np.inf, rng.uniform(0.2, 3, n))
    p["attenuation_colour"] = rng.uniform(0.05, 1, (n, 3))
    with Renderer(w, h) as r:
        r.set_ggx_lut(ggx_lut)
        r.set_opaque_frame(bits)
        r.generate_mips()
        got = r.eval_ibl_volume_refraction(pv, p)
    ref = oracle.eval_ibl_volume_refraction(pv, p, levels, ggx_lut)
    assert rel_l2(got, ref) < 2e-5
    assert np.median(np.abs(got - ref) / (np.abs(ref) + 1e-3)) < 2e-6


# ------------------------------------------------------------------------------ K5 mip chain (bit-exact)
@pytest.mark.parametrize("size", [(512, 512), (1920, 1080), (37, 23), (100, 60), (64, 2), (2, 2), (130, 66), (1024, 8)])
def test_mip_chain_bit_exact(oracle, size):
    w, h = size
    img = scenes.procedural_opaque_frame(w, h, seed=0xABC0 + w)
    img[::7, ::5, :3] *= 100.0   # a few large values so fp16 rounding at several exponents is exercised
    bits = oracle.f16_bits(img)
    levels = oracle.build_pyramid(bits)
    with Renderer(w, h) as r:
        assert r.mip_levels() == len(levels)
        r.set_opaque_frame(bits)
        r.generate_mips()
        for l, ref in enumerate(levels):
            got = r.read_pyramid_level(l)
            assert got.shape == ref.shape
            np.testing.assert_array_equal(got, ref, err_msg=f"level {l} of {w}x{h}")
        # idempotence / re-arming of the single-pass ticket: a second launch gives the same bytes
        r.generate_mips()
        np.testing.assert_array_equal(r.read_pyramid_level(len(levels) - 1), levels[-1])


# ------------------------------------------------------------------------------ config 1: synthetic G-buffer, transmission
@pytest.mark.parametrize("size,roughness", [(512, 0.25), (96, 0.6), (131, 0.1)])
def test_config1_transmission(oracle, ggx_lut, size, roughness):
    s = scenes.config1(size, roughness)
    cam = s["camera"]
    pc = cam.push_constants()
    n_cl = host.NUM_CLUSTERS
    counts = np.zeros(n_cl, np.uint32)
    indices = np.zeros(n_cl * abi.TR_MAX_LIGHTS_PER_CLUSTER, np.uint32)
    bits = oracle.f16_bits(s["opaque"])
    levels = oracle.build_pyramid(bits)
    sc = oracle_scene(pc, s["uniforms"], s["materials"], s["lights"], counts, indices)
    zero32 = np.zeros((size, size, 4), f32)
    zero16 = np.zeros((size, size, 4), np.uint16)
    ref32, ref16 = oracle.shade_transmission_frame(s["gbuffer"], sc, levels, ggx_lut, zero32, zero16)
    with Renderer(size, size, f32_debug=True) as r:
        gpu_setup(r, ggx_lut, s["uniforms"], s["materials"], s["lights"])
        r.set_gbuffer(abi.TR_LAYER_TRANSMISSIVE, s["gbuffer"])
        r.set_opaque_frame(bits)
        r.generate_mips()
        r.shade_transmission(pc)
        got32, got16 = r.read_hdr_f32(), r.read_hdr()
        r.tonemap(host.default_tonemap_params())
        srgb = r.read_srgb8()
    e32 = rel_l2(got32[..., :3], ref32[..., :3])
    e16 = rel_l2(oracle.f16_to_f32(got16)[..., :3], oracle.f16_to_f32(ref16)[..., :3])
    print(f"config1 {size}^2 r={roughness}: rel-L2 fp32 {e32:.2e}, fp16 {e16:.2e}")
    assert e32 < REL_L2_TOL and e16 < REL_L2_TOL
    ref_srgb = oracle.tonemap_frame(ref16, host.default_tonemap_params())
    assert np.max(np.abs(srgb.astype(int) - ref_srgb.astype(int))) <= SRGB_TOL


# ------------------------------------------------------------------------------ opaque + transmission over ray-cast spheres
def _sphere_layers(w, h, seed):
    cam = scenes.Camera(w, h, (0.0, 3.0, 6.0), 0.0, -15.0)
    rng = np.random.default_rng(seed)
    n_o, n_t = 40, 10
    co = np.stack([rng.uniform(-4, 4, n_o), rng.uniform(0.3, 3.5, n_o), rng.uniform(-8, 0, n_o)], -1)
    ro = rng.uniform(0.3, 0.8, n_o)
    ct = np.stack([rng.uniform(-3, 3, n_t), rng.uniform(1.0, 3.0, n_t), rng.uniform(0.5, 2.5, n_t)], -1)
    rt = rng.uniform(0.3, 0.7, n_t)
    mats = np.concatenate([scenes.hashed_materials(n_o, seed), scenes.hashed_materials(n_t, seed ^ 5, True, (0.15, 0.5))])
    g0 = scenes.raycast_spheres(cam, co, ro, np.arange(n_o))
    g1 = scenes.raycast_spheres(cam, ct, rt, n_o + np.arange(n_t), scale_plane=True)
    # the transmissive layer only survives where it is nearer than the opaque layer (depth GREATER, reversed-Z)
    keep = g1["depth"] > g0["depth"]
    g1["depth"] = np.where(keep, g1["depth"], 0).astype(f32)
    g1["material_id"] = np.where(keep, g1["material_id"], 0xFFFFFFFF).astype(np.uint32)
    g1["scale"] = (1.0 + 0.5 * rng.random((h, w))).astype(f32)
    return cam, mats, g0, g1


@pytest.mark.parametrize("size,n_lights,spot", [((640, 360), 4, False), ((333, 187), 24, True), ((1920, 1080), 4, False)])
def test_shade_path_spheres(oracle, ggx_lut, size, n_lights, spot):
    w, h = size
    cam, mats, g0, g1 = _sphere_layers(w, h, 7 + n_lights)
    uniforms = host.make_uniforms(w, h)
    lights = scenes.config2_lights() if n_lights == 4 else scenes.hashed_point_lights(
        n_lights, 99, box=((-6, 0.5, -9), (6, 5, 4)), intensity=(2.0, 30.0))
    if spot:
        lights = np.concatenate([lights, host.light_new_spot((0, 4, 0), (1, 1, 0.5), 50.0, (0.2, -0.9, -0.3), 0.7, 0.8)])
    pc = cam.push_constants()
    aabbs, counts, indices = oracle_cluster_lights(oracle, cam, uniforms, lights)
    sc = oracle_scene(pc, uniforms, mats, lights, counts, indices)
    o32, o16 = oracle.shade_opaque_frame(g0, sc)
    levels = oracle.build_pyramid(o16)
    t32, t16 = oracle.shade_transmission_frame(g1, sc, levels, ggx_lut, o32, o16)
    ref_srgb = oracle.tonemap_frame(t16, host.default_tonemap_params())

    with Renderer(w, h, f32_debug=True) as r:
        gpu_setup(r, ggx_lut, uniforms, mats, lights)
        r.build_clusters(cam.write_cluster_data())
        r.assign_lights(cam.assign_lights())
        # discrete stage: cluster AABBs and ordered light lists bit-exact
        got_aabbs = r.read_cluster_aabbs(len(aabbs))
        assert got_aabbs.tobytes() == aabbs.tobytes()
        gc, gi = r.read_cluster_lights(len(aabbs))
        np.testing.assert_array_equal(gc, counts)
        mask = np.arange(abi.TR_MAX_LIGHTS_PER_CLUSTER)[None, :] < counts[:, None]
        np.testing.assert_array_equal(gi.reshape(-1, 128)[mask], indices.reshape(-1, 128)[mask])
        assert counts.max() > 0

        r.set_gbuffer(abi.TR_LAYER_OPAQUE, g0)
        r.set_gbuffer(abi.TR_LAYER_TRANSMISSIVE, g1)
        r.shade_opaque(pc)
        go32, go16 = r.read_hdr_f32(), r.read_hdr()
        np.testing.assert_array_equal(r.read_pyramid_level(0), go16)   # both targets get the same value (lib.rs:247-248)
        r.generate_mips()
        r.shade_transmission(pc)
        gt32, gt16 = r.read_hdr_f32(), r.read_hdr()
        r.tonemap(host.default_tonemap_params())
        srgb = r.read_srgb8()

    e_o32 = rel_l2(go32[..., :3], o32[..., :3])
    e_o16 = rel_l2(oracle.f16_to_f32(go16)[..., :3], oracle.f16_to_f32(o16)[..., :3])
    e_t32 = rel_l2(gt32[..., :3], t32[..., :3])
    e_t16 = rel_l2(oracle.f16_to_f32(gt16)[..., :3], oracle.f16_to_f32(t16)[..., :3])
    print(f"spheres {w}x{h} L={len(lights)}: opaque rel-L2 fp32 {e_o32:.2e} fp16 {e_o16:.2e}; "
          f"final fp32 {e_t32:.2e} fp16 {e_t16:.2e}")
    assert max(e_o32, e_o16, e_t32, e_t16) < REL_L2_TOL
    assert (g1["depth"] > 0).mean() > 0.02 and (g0["depth"] > 0).mean() > 0.1
    assert np.max(np.abs(srgb.astype(int) - ref_srgb.astype(int))) <= SRGB_TOL
    # alpha is exactly 1 everywhere and empty pixels keep the clear colour (main.rs:1592-1602)
    assert (go16[..., 3] == 0x3C00).all()
    empty = g0["depth"] == 0
    assert (go16[empty][:, :3] == 0).all()


def test_bands_equal_full_frame(oracle, ggx_lut):
    """Shading the frame as 3 ragged bands gives the same bytes as one pass (tiling independence)."""
    w, h = 322, 181
    cam, mats, g0, g1 = _sphere_layers(w, h, 21)
    uniforms = host.make_uniforms(w, h)
    lights = scenes.config2_lights()
    pc = cam.push_constants()
    outs = []
    for bands in ([(0, h)], [(0, 61), (61, 120), (120, h)]):
        with Renderer(w, h) as r:
            gpu_setup(r, ggx_lut, uniforms, mats, lights)
            r.build_clusters(cam.write_cluster_data())
            r.assign_lights(cam.assign_lights())
            r.set_gbuffer(0, g0)
            r.set_gbuffer(1, g1)
            for (y0, y1) in bands:
                r.set_band(y0, y1)
                r.shade_opaque(pc)
            r.generate_mips()
            for (y0, y1) in bands:
                r.set_band(y0, y1)
                r.shade_transmission(pc)
            outs.append(r.read_hdr())
    np.testing.assert_array_equal(outs[0], outs[1])


# ------------------------------------------------------------------------------ K1 cull + demux (bit-exact)
@pytest.mark.parametrize("n_inst", [1, 255, 256, 257, 10000, 100003])
def test_cull_bit_exact(oracle, n_inst):
    s = scenes.instanced_scene(640, 360, n_instances=n_inst, n_lights=0, seed=0x5EED0004 + n_inst)
    cam = s["camera"]
    cpc = cam.culling()
    counts, visible = oracle.frustum_culling(s["instances"], s["primitives"], cpc)
    draws, dcounts = oracle.demultiplex_draws(s["primitives"], counts)
    with Renderer(64, 64) as r:
        r.set_instances(s["instances"])
        r.set_primitives(s["primitives"])
        for _ in range(2):   # twice: the per-frame state block must re-arm
            r.cull(cpc)
            np.testing.assert_array_equal(r.read_visible_instances(), visible)
            np.testing.assert_array_equal(r.read_instance_counts(len(s["primitives"])), counts)
            for b in range(4):
                got = r.read_draws(b)
                assert got.tobytes() == draws[b].tobytes()
    if n_inst >= 10000:
        assert 0.2 * n_inst < len(visible) < 0.8 * n_inst


def test_cull_adversarial_boundary(oracle):
    """Instances placed within a few ulps of the cull planes: the visibility bits must still agree."""
    cam = scenes.Camera(640, 360, (0.3, 1.0, -2.0), 30.0, -10.0)
    cpc = cam.culling()
    rng = np.random.default_rng(5)
    n = 20000
    prims = np.zeros(1, dtype=abi.primitive_info)
    prims["packed_bounding_sphere"] = (0.1, 0.2, -0.1, 1.0)
    prims["index_count"] = 3
    inst = np.zeros(n, dtype=abi.instance)
    inst["rotation"] = (0, 0, 0, 1)
    # put the sphere centres on the near-test boundary: view-space z' + r == z_near, then jitter by ulps
    view = cam.view.astype(np.float64)
    fwd = -view[2, :3]
    base = cam.position.astype(np.float64)
    lateral = rng.uniform(-0.3, 0.3, (n, 2))  # inside the side planes, so the near test decides
    scale = rng.uniform(0.5, 2.0, n)
    centre = base + fwd[None, :] * (0.01 - scale)[:, None] + view[0, :3][None, :] * lateral[:, :1] + view[1, :3][None, :] * lateral[:, 1:]
    t = centre - scale[:, None] * np.array([0.1, 0.2, -0.1])
    inst["translation_and_scale"][:, :3] = t
    inst["translation_and_scale"][:, 3] = scale
    ulps = rng.integers(-3, 4, (n, 3)).astype(np.int32)
    tv = inst["translation_and_scale"][:, :3].copy().view(np.int32)
    inst["translation_and_scale"][:, :3] = (tv + ulps).view(f32)
    counts, visible = oracle.frustum_culling(inst, prims, cpc)
    assert 0.2 * n < len(visible) < 0.8 * n
    with Renderer(64, 64) as r:
        r.set_instances(inst)
        r.set_primitives(prims)
        r.cull(cpc)
        np.testing.assert_array_equal(r.read_visible_instances(), visible)


def test_cluster_index_adversarial(oracle, ggx_lut):
    """Pixels whose depth sits on cluster-slice boundaries: light lists differ across the boundary, so a
    single mis-sliced pixel shows up as a large error."""
    w, h = 256, 144
    cam = scenes.Camera(w, h, (0.0, 2.0, 5.0), 0.0, -5.0)
    uniforms = host.make_uniforms(w, h)
    zn, zf = float(host.Z_NEAR), float(host.Z_FAR)
    a = zn / (zf - zn)
    b = zf * a
    rng = np.random.default_rng(3)
    # slice boundaries: dist = near * (far/near)^(k/16); depth = b/dist - a; jitter by a few ulps
    k = rng.integers(6, 14, (h, w))
    dist = zn * (zf / zn) ** (k / 16.0)
    depth = (b / dist - a).astype(f32)
    depth = (depth.view(np.int32) + rng.integers(-4, 5, (h, w)).astype(np.int32)).view(f32)
    n = np.zeros((h, w, 3), f32)
    n[..., 1] = 0.6
    n[..., 2] = 0.8
    g0 = dict(depth=depth, normal=n, uv=None, material_id=np.zeros((h, w), np.uint32), scale=None, position=None)
    mats = abi.default_material(1)
    mats["metallic_factor"] = 0.0
    mats["roughness_factor"] = 0.5
    lights = scenes.hashed_point_lights(48, 1234, box=((-20, 0, -60), (20, 10, 5)), intensity=(5.0, 40.0))
    pc = cam.push_constants()
    _, counts, indices = oracle_cluster_lights(oracle, cam, uniforms, lights)
    sc = oracle_scene(pc, uniforms, mats, lights, counts, indices)
    o32, o16 = oracle.shade_opaque_frame(g0, sc)
    with Renderer(w, h, f32_debug=True) as r:
        gpu_setup(r, None, uniforms, mats, lights)
        r.set_cluster_lights(counts, indices)
        r.set_gbuffer(0, g0)
        r.shade_opaque(pc)
        got = r.read_hdr_f32()
    err = np.abs(got[..., :3] - o32[..., :3]) / (np.abs(o32[..., :3]) + 1e-6)
    assert err.max() < 1e-3, "a pixel landed in the wrong cluster slice"
    assert rel_l2(got[..., :3], o32[..., :3]) < REL_L2_TOL


# ------------------------------------------------------------------------------ K7 tonemap
def test_tonemap_srgb8(oracle):
    rng = np.random.default_rng(8)
    w, h = 640, 361
    hdr = np.ones((h, w, 4), f32)
    hdr[..., :3] = np.exp2(rng.uniform(-12, 6, (h, w, 3)))
    hdr[:10, :, :3] = 0.0
    hdr[10:20, :, 1:3] = 0.0
    bits = oracle.f16_bits(hdr)
    params = host.default_tonemap_params()
    ref = oracle.tonemap_frame(bits, params)
    with Renderer(w, h) as r:
        r.set_hdr(bits)
        r.tonemap(params)
        got = r.read_srgb8()
    diff = np.abs(got.astype(int) - ref.astype(int))
    assert diff.max() <= SRGB_TOL
    assert (diff > 0).mean() < 0.02
    assert (got[:10, :, :3] == 0).all() and (got[..., 3] == 255).all()


# ------------------------------------------------------------------------------ K3 visibility (bit-exact) and whole frames
def _frame_scene(kind, w, h):
    if kind == "grid":
        return scenes.sphere_grid_scene(w, h, transmissive_knot=True)
    if kind == "instanced":
        return scenes.instanced_scene(w, h, n_instances=3000, n_lights=32)
    raise ValueError(kind)


def _oracle_frame(oracle, lut, s, y0=0, y1=None):
    cam = s["camera"]
    pc = cam.push_constants()
    counts, visible = oracle.frustum_culling(s["instances"], s["primitives"], cam.culling())
    g0, g1 = oracle.visibility(s["mesh"], s["instances"], s["primitives"], visible, pc, y0, y1)
    _, cc, ci = oracle_cluster_lights(oracle, cam, s["uniforms"], s["lights"])
    sc = oracle_scene(pc, s["uniforms"], s["materials"], s["lights"], cc, ci)
    o32, o16 = oracle.shade_opaque_frame(g0, sc, y0, y1)
    return dict(visible=visible, g0=g0, g1=g1, scene=sc, o32=o32, o16=o16)


def _upload_scene(r, lut, s):
    gpu_setup(r, lut, s["uniforms"], s["materials"], s["lights"])
    r.set_instances(s["instances"])
    r.set_primitives(s["primitives"])
    m = s["mesh"]
    r.set_mesh(m["positions"], m["normals"], m["uvs"], m["indices"])
    r.build_clusters(s["camera"].write_cluster_data())


@pytest.mark.parametrize("kind,size,tile_edge,split,front", [("grid", (640, 360), None, None, None), ("instanced", (480, 270), None, None, None),
                                                             ("instanced", (333, 187), None, None, None), ("instanced", (480, 270), 64, 0, None),
                                                             ("grid", (640, 360), 64, 0, None), ("instanced", (960, 540), 32, None, None),
                                                             ("instanced", (960, 540), 64, 1, None), ("grid", (640, 360), 64, 1, None),
                                                             ("instanced", (960, 540), None, None, "TR_NO_CHUNK_CULL"),
                                                             ("instanced", (960, 540), None, None, "TR_NO_BLOCK_ENTRY")])
def test_visibility_bit_exact(oracle, ggx_lut, kind, size, tile_edge, split, front, monkeypatch):
    """tile_edge forces the rasteriser's 64- or 32-pixel tile instantiation (it otherwise follows the frame size, so the
    small test frames would only ever run the 32-pixel one and the 4K benchmark only the 64-pixel one); split forces the
    quadrant jobs of heavy tiles on (a many-GPU band's path) or off; front switches one shortcut of the binning front end
    off (the chunk-sphere test against the frame / band planes, the 256-triangle entry table), so both forms stay pinned."""
    if front is not None:
        monkeypatch.setenv(front, "1")
    if tile_edge is not None:
        monkeypatch.setenv("TR_TILE_EDGE", str(tile_edge))
    if split is not None:
        monkeypatch.setenv("TR_TILE_SPLIT", str(split))
    w, h = size
    s = _frame_scene(kind, w, h)
    ref = _oracle_frame(oracle, ggx_lut, s)
    cam = s["camera"]
    with Renderer(w, h) as r:
        _upload_scene(r, ggx_lut, s)
        for _ in range(2):   # second frame exercises the in-kernel clear of the visibility words
            r.cull(cam.culling())
            r.visibility(cam.push_constants())
            for layer, g in ((0, ref["g0"]), (1, ref["g1"])):
                got = r.read_gbuffer(layer)
                for k in ("depth", "normal", "uv", "material_id") + (("scale",) if layer == 1 else ()):
                    a, b = got[k], np.asarray(g[k]).reshape(got[k].shape)
                    assert a.tobytes() == b.tobytes(), f"layer {layer} plane {k}: {(a != b).sum()} values differ"
    assert (ref["g0"]["depth"] > 0).mean() > 0.2 and (ref["g1"]["depth"] > 0).mean() > 0.01


@pytest.mark.parametrize("kind,size", [("grid", (640, 360)), ("instanced", (480, 270))])
def test_full_frame(oracle, ggx_lut, kind, size):
    """record() order end to end through tr_frame vs the oracle chain."""
    w, h = size
    s = _frame_scene(kind, w, h)
    ref = _oracle_frame(oracle, ggx_lut, s)
    levels = oracle.build_pyramid(ref["o16"])
    t32, t16 = oracle.shade_transmission_frame(ref["g1"], ref["scene"], levels, ggx_lut, ref["o32"], ref["o16"])
    params = host.default_tonemap_params()
    ref_srgb = oracle.tonemap_frame(t16, params)
    cam = s["camera"]
    with Renderer(w, h, f32_debug=True) as r:
        _upload_scene(r, ggx_lut, s)
        r.enable_timing(True)
        r.frame(cam.frame_params(params))
        times = r.frame_times()
        got32, got16, srgb = r.read_hdr_f32(), r.read_hdr(), r.read_srgb8()
        for l, lv in enumerate(levels):   # GPU mips of the GPU opaque frame vs oracle mips of the oracle frame
            assert rel_l2(oracle.f16_to_f32(r.read_pyramid_level(l))[..., :3], oracle.f16_to_f32(lv)[..., :3]) < REL_L2_TOL
    e32 = rel_l2(got32[..., :3], t32[..., :3])
    e16 = rel_l2(oracle.f16_to_f32(got16)[..., :3], oracle.f16_to_f32(t16)[..., :3])
    print(f"frame {kind} {w}x{h}: rel-L2 fp32 {e32:.2e} fp16 {e16:.2e}; times {times}")
    assert e32 < REL_L2_TOL and e16 < REL_L2_TOL
    d = np.abs(srgb.astype(int) - ref_srgb.astype(int))
    assert d.max() <= SRGB_TOL, f"{(d > SRGB_TOL).sum()} channels off by more than {SRGB_TOL}/255"
    assert times["total_ms"] > 0


# ------------------------------------------------------------------------------ edge cases and error behaviour
def test_light_list_overflow_is_clamped(oracle):
    """More than MAX_LIGHTS_PER_CLUSTER (128) lights reach one cluster: the reference's append would run into the next
    cluster's slice (shader/src/lib.rs:640-644); both sides keep the 128 lowest ids instead."""
    w, h = 128, 72
    cam = scenes.Camera(w, h, (0.0, 2.0, 5.0), 0.0, -5.0)
    uniforms = host.make_uniforms(w, h)
    lights = scenes.hashed_point_lights(200, 77, box=((-1, 1, 0), (1, 3, 2)), intensity=(40.0, 50.0))
    aabbs, counts, indices = oracle_cluster_lights(oracle, cam, uniforms, lights)
    assert counts.max() == abi.TR_MAX_LIGHTS_PER_CLUSTER
    with Renderer(w, h) as r:
        gpu_setup(r, None, uniforms, abi.default_material(1), lights)
        r.build_clusters(cam.write_cluster_data())
        r.assign_lights(cam.assign_lights())
        gc, gi = r.read_cluster_lights(len(aabbs))
    np.testing.assert_array_equal(gc, counts)
    used = np.arange(abi.TR_MAX_LIGHTS_PER_CLUSTER)[None, :] < counts[:, None]
    np.testing.assert_array_equal(gi.reshape(-1, abi.TR_MAX_LIGHTS_PER_CLUSTER)[used], indices.reshape(-1, abi.TR_MAX_LIGHTS_PER_CLUSTER)[used])


def test_empty_view_and_resize(oracle, ggx_lut):
    """Camera looking away from everything: nothing visible, the frame is the clear colour; then the swapchain-resize
    path (src/main.rs:996-1166) and a normal frame at the new size."""
    s = scenes.sphere_grid_scene(320, 180, transmissive_knot=True)
    away = scenes.Camera(320, 180, (0.0, 3.0, 6.0), 180.0, 60.0)
    with Renderer(320, 180) as r:
        _upload_scene(r, ggx_lut, s)
        r.build_clusters(away.write_cluster_data())
        r.frame(away.frame_params(host.default_tonemap_params()))
        assert len(r.read_visible_instances()) <= 1   # only the ground quad's huge bounding sphere survives the cull
        hdr = oracle.f16_to_f32(r.read_hdr())
        assert (hdr[..., :3] == 0).all() and (hdr[..., 3] == 1).all()
        assert (r.read_gbuffer(0)["depth"] == 0).all() and (r.read_gbuffer(1)["depth"] == 0).all()
        w, h = 200, 120
        r.resize(w, h)
        s2 = scenes.sphere_grid_scene(w, h, transmissive_knot=True)
        cam = s2["camera"]
        r.set_uniforms(s2["uniforms"])
        r.build_clusters(cam.write_cluster_data())
        r.frame(cam.frame_params(host.default_tonemap_params()))
        got = r.read_hdr()
        assert got.shape == (h, w, 4)
        ref = _oracle_frame(oracle, ggx_lut, s2)
        levels = oracle.build_pyramid(ref["o16"])
        _, t16 = oracle.shade_transmission_frame(ref["g1"], ref["scene"], levels, ggx_lut, ref["o32"], ref["o16"])
        assert rel_l2(oracle.f16_to_f32(got)[..., :3], oracle.f16_to_f32(t16)[..., :3]) < REL_L2_TOL


def test_error_behaviour():
    """The boundary never ignores what it does not implement and enforces call order (include/tr_abi.h)."""
    from transmission_renderer_b200 import TrError
    cam = scenes.Camera(64, 64)
    with Renderer(64, 64) as r:
        m = abi.default_material(1)
        m["textures"][0, 0] = 500
        with pytest.raises(TrError) as e:
            r.set_materials(m)
        assert e.value.status == -1                                   # TR_ERR_INVALID_ARG: image index beyond MAX_IMAGES
        p = np.zeros(1, dtype=abi.primitive_info)
        p["draw_buffer_index"] = 4
        with pytest.raises(TrError) as e:
            r.set_primitives(p)
        assert e.value.status == -1                                   # there are four draw buffers
        u = host.make_uniforms(64, 64)
        u["debug_clusters"] = 1
        with pytest.raises(TrError) as e:
            r.set_uniforms(u)
        assert e.value.status == -2
        with pytest.raises(TrError) as e:
            r.shade_opaque(cam.push_constants())
        assert e.value.status == -6                                   # TR_ERR_STATE: uniforms / G-buffer missing
        r.set_uniforms(host.make_uniforms(64, 64))
        r.set_materials(abi.default_material(1))
        pc = cam.push_constants()
        pc["acceleration_structure_address"] = 1
        with pytest.raises(TrError) as e:
            r.shade_opaque(pc)
        assert e.value.status == -1                                   # not a handle of tr_build_acceleration_structures
        bad = scenes.Camera(32, 32).push_constants()
        with pytest.raises(TrError) as e:
            r.shade_opaque(bad)
        assert e.value.status == -1                                   # TR_ERR_INVALID_ARG: framebuffer size mismatch
        with pytest.raises(TrError) as e:
            r.generate_mips()
        assert e.value.status == -6
    with pytest.raises(TrError):
        Renderer(0, 10)


# ------------------------------------------------------------------------------ row N2: texture-mapped materials, normal mapping
def _textured_reference(oracle, lut, s):
    cam = s["camera"]
    pc = cam.push_constants()
    _, visible = oracle.frustum_culling(s["instances"], s["primitives"], cam.culling())
    g0, g1 = oracle.visibility(s["mesh"], s["instances"], s["primitives"], visible, pc, derivatives=True,
                               materials=s["materials"], textures=s["textures"])
    _, cc, ci = oracle_cluster_lights(oracle, cam, s["uniforms"], s["lights"])
    sc = oracle_scene(pc, s["uniforms"], s["materials"], s["lights"], cc, ci)
    sc["textures"] = s["textures"]
    o32, o16 = oracle.shade_opaque_frame(g0, sc)
    levels = oracle.build_pyramid(o16)
    t32, t16 = oracle.shade_transmission_frame(g1, sc, levels, lut, o32, o16)
    return dict(g0=g0, g1=g1, o32=o32, o16=o16, t32=t32, t16=t16)


@pytest.mark.parametrize("size", [(640, 360), (333, 187)])
def test_textured_frame(oracle, ggx_lut, size):
    """Every texture slot the shaders read (diffuse, metallic-roughness, normal map, emissive, transmission, thickness,
    specular, specular colour), implicit level of detail from the uv differences, repeat addressing, normal mapping
    through the cotangent frame — whole frames against the oracle; the derivative planes of the G-buffer bit for bit."""
    w, h = size
    s = scenes.textured_sphere_scene(w, h)
    ref = _textured_reference(oracle, ggx_lut, s)
    cam = s["camera"]
    with Renderer(w, h, f32_debug=True) as r:
        r.set_textures(s["textures"])
        _upload_scene(r, ggx_lut, s)
        r.frame(cam.frame_params(host.default_tonemap_params()))
        for layer, g in ((0, ref["g0"]), (1, ref["g1"])):
            got = r.read_gbuffer(layer, derivatives=True)
            for k in ("depth", "uv", "duv", "ddepth"):
                assert got[k].tobytes() == np.asarray(g[k]).tobytes(), f"layer {layer} plane {k}: {(got[k] != g[k]).sum()} values differ"
        got32 = r.read_hdr_f32()
        got_o16 = r.read_pyramid_level(0)
    duv = ref["g0"]["duv"][ref["g0"]["depth"] > 0]
    assert np.abs(duv).max() > 1e-3                                           # the level of detail is really exercised
    e_o = rel_l2(oracle.f16_to_f32(got_o16)[..., :3], oracle.f16_to_f32(ref["o16"])[..., :3])
    e_t = rel_l2(got32[..., :3], ref["t32"][..., :3])
    print(f"textured {w}x{h}: opaque fp16 rel-L2 {e_o:.2e}, final fp32 rel-L2 {e_t:.2e}")
    assert e_o < REL_L2_TOL and e_t < REL_L2_TOL
    # the textures matter: the same frame with the bindings removed is far away
    plain = dict(s, materials=s["materials"].copy())
    plain["materials"]["textures"] = -1
    with Renderer(w, h, f32_debug=True) as r:
        _upload_scene(r, ggx_lut, plain)
        r.frame(cam.frame_params(host.default_tonemap_params()))
        untextured = r.read_hdr_f32()
    assert rel_l2(untextured[..., :3], ref["t32"][..., :3]) > 0.05


# ------------------------------------------------------------------------------ row N3: alpha-clip draw buffers
@pytest.mark.parametrize("size", [(640, 360), (301, 170)])
def test_alpha_clip_frame(oracle, ggx_lut, size):
    """Draw buffers 1 and 3: fragments whose diffuse alpha (factor x texture) is below the cutoff are killed in the depth
    pre-pass, so what lies behind shows through.  G-buffer planes bit for bit, whole frame within tolerance."""
    w, h = size
    s = scenes.alpha_clip_scene(w, h)
    ref = _textured_reference(oracle, ggx_lut, s)
    cam = s["camera"]
    with Renderer(w, h, f32_debug=True) as r:
        r.set_textures(s["textures"])
        _upload_scene(r, ggx_lut, s)
        counts, visible = oracle.frustum_culling(s["instances"], s["primitives"], cam.culling())
        draws, dcounts = oracle.demultiplex_draws(s["primitives"], counts)
        r.frame(cam.frame_params(host.default_tonemap_params()))
        for b in range(4):
            assert r.read_draws(b).tobytes() == draws[b].tobytes()
        assert dcounts[1] > 0 and dcounts[3] > 0
        for layer, g in ((0, ref["g0"]), (1, ref["g1"])):
            got = r.read_gbuffer(layer, derivatives=True)
            for k in ("depth", "normal", "uv", "material_id", "duv", "ddepth"):
                a, b_ = got[k], np.asarray(g[k]).reshape(got[k].shape)
                assert a.tobytes() == b_.tobytes(), f"layer {layer} plane {k}: {(a != b_).sum()} values differ"
        got32 = r.read_hdr_f32()
    e_t = rel_l2(got32[..., :3], ref["t32"][..., :3])
    print(f"alpha clip {w}x{h}: final fp32 rel-L2 {e_t:.2e}")
    assert e_t < REL_L2_TOL
    # the alpha test really removes fragments: without materials (no clipping) the oracle's opaque layer differs
    _, vis2 = oracle.frustum_culling(s["instances"], s["primitives"], cam.culling())
    g0_solid, g1_solid = oracle.visibility(s["mesh"], s["instances"], s["primitives"], vis2, cam.push_constants())
    assert (g0_solid["material_id"] != ref["g0"]["material_id"]).mean() > 0.01
    assert (g1_solid["depth"] != ref["g1"]["depth"]).mean() > 0.002


# ------------------------------------------------------------------------------ row N4: an ingested glTF asset
def test_ingested_gltf_frame(oracle, ggx_lut, tmp_path):
    """A glTF file (node hierarchy, all four draw buffers, textures bound through base colour / metallic-roughness /
    normal / specular slots, KHR transmission + volume + ior) goes through gltf_ingest (mirror of src/model_loading.rs)
    into the C ABI; G-buffer planes bit for bit, whole frame within tolerance against the oracle on the same arrays."""
    from test_gltf_ingest import _asset
    from transmission_renderer_b200 import gltf_ingest
    path, _ = _asset(tmp_path)
    w, h = 640, 360
    s = gltf_ingest.finish(gltf_ingest.load_gltf(path))
    s.update(camera=scenes.Camera(w, h, (0.0, 3.0, 6.0), 0.0, -15.0), lights=scenes.config2_lights(),
             uniforms=host.make_uniforms(w, h))
    ref = _textured_reference(oracle, ggx_lut, s)
    cam = s["camera"]
    with Renderer(w, h, f32_debug=True) as r:
        r.set_textures(s["textures"])
        _upload_scene(r, ggx_lut, s)
        r.frame(cam.frame_params(host.default_tonemap_params()))
        for layer, g in ((0, ref["g0"]), (1, ref["g1"])):
            got = r.read_gbuffer(layer, derivatives=True)
            for k in ("depth", "normal", "uv", "material_id", "duv", "ddepth"):
                a, b_ = got[k], np.asarray(g[k]).reshape(got[k].shape)
                assert a.tobytes() == b_.tobytes(), f"layer {layer} plane {k}: {(a != b_).sum()} values differ"
        got32 = r.read_hdr_f32()
    assert set(np.unique(ref["g0"]["material_id"][ref["g0"]["depth"] > 0])) == {0, 1, 4}
    assert set(np.unique(ref["g1"]["material_id"][ref["g1"]["depth"] > 0])) == {2, 3}
    e_t = rel_l2(got32[..., :3], ref["t32"][..., :3])
    print(f"ingested glTF {w}x{h}: final fp32 rel-L2 {e_t:.2e}")
    assert e_t < REL_L2_TOL


# ------------------------------------------------------------------------------ adversarial shading inputs
def test_random_gbuffer_stress(oracle, ggx_lut):
    """Random G-buffer pixels that hit the ill-conditioned corners of the lobes on purpose: normals facing away from the
    viewer (n.v clamped to EPSILON), grazing lights, roughness down to 0.05, lights a few centimetres from the surface.
    Both shading passes against the oracle: relative L2 of the frame and the share of pixels off by more than 1e-3."""
    w, h = 256, 192
    rng = np.random.default_rng(11)
    cam = scenes.Camera(w, h, (0.0, 2.0, 5.0), 0.0, -5.0)
    uniforms = host.make_uniforms(w, h)
    pc = cam.push_constants()
    # positions: unproject random depths between 1.5 m and 12 m
    dist = rng.uniform(1.5, 12.0, (h, w))
    zn, zf = float(host.Z_NEAR), float(host.Z_FAR)
    a = zn / (zf - zn)
    depth = (zf * a / dist - a).astype(f32)
    n = _rand_unit(rng, h * w).reshape(h, w, 3).astype(f32) * rng.uniform(0.5, 2.0, (h, w, 1)).astype(f32)  # un-normalised, any facing
    n_mat = 48
    mats = scenes.hashed_materials(n_mat, 21, roughness_range=(0.05, 1.0))
    tmats = scenes.hashed_materials(n_mat, 22, True, (0.05, 0.6))
    materials = np.concatenate([mats, tmats])
    mid = rng.integers(0, n_mat, (h, w)).astype(np.uint32)
    g0 = dict(depth=depth, normal=n, uv=None, material_id=mid, scale=None, position=None)
    g1 = dict(depth=depth, normal=n, uv=None, material_id=(mid + n_mat).astype(np.uint32),
              scale=rng.uniform(0.5, 2.0, (h, w)).astype(f32), position=None)
    lights = scenes.hashed_point_lights(40, 99, box=((-6, 0.2, -8), (6, 5, 4)), intensity=(2.0, 30.0))
    _, counts, indices = oracle_cluster_lights(oracle, cam, uniforms, lights)
    assert counts.max() > 8
    sc = oracle_scene(pc, uniforms, materials, lights, counts, indices)
    o32, o16 = oracle.shade_opaque_frame(g0, sc)
    levels = oracle.build_pyramid(o16)
    t32, _ = oracle.shade_transmission_frame(g1, sc, levels, ggx_lut, o32, o16)
    with Renderer(w, h, f32_debug=True) as r:
        gpu_setup(r, ggx_lut, uniforms, materials, lights)
        r.set_cluster_lights(counts, indices)
        r.set_gbuffer(0, g0)
        r.set_gbuffer(1, g1)
        r.shade_opaque(pc)
        got_o = r.read_hdr_f32()
        r.generate_mips()
        r.shade_transmission(pc)
        got_t = r.read_hdr_f32()
    for name, got, ref in (("opaque", got_o, o32), ("transmission", got_t, t32)):
        e = rel_l2(got[..., :3], ref[..., :3])
        ok = np.isfinite(ref[..., :3]) & np.isfinite(got[..., :3])
        rel = np.abs(got[..., :3] - ref[..., :3])[ok] / (np.abs(ref[..., :3])[ok] + 1e-3)
        bad = float((rel > 1e-3).mean())
        print(f"stress {name}: rel-L2 {e:.2e}, share of values off by > 1e-3: {bad:.2e}, worst {rel.max():.2e}")
        assert e < REL_L2_TOL and bad < 1e-4


def test_more_lights_than_the_shared_table(oracle, ggx_lut):
    """1 200 lights: more than the 768-entry shared-memory light table of the shading kernels, so the launch takes the
    global-memory light path (the huge far clusters overflow their 128-entry lists, which both sides clamp alike)."""
    w, h = 320, 180
    cam = scenes.Camera(w, h, (0.0, 3.0, 6.0), 0.0, -15.0)
    uniforms = host.make_uniforms(w, h)
    lights = scenes.hashed_point_lights(1200, 4242, box=((-40, 0.3, -60), (40, 8, 10)), intensity=(0.2, 1.5))
    rng = np.random.default_rng(2)
    centres = np.stack([rng.uniform(-4, 4, 12), rng.uniform(0.5, 3.0, 12), rng.uniform(-6, 1, 12)], -1)
    g0 = scenes.raycast_spheres(cam, centres, rng.uniform(0.4, 0.9, 12), np.arange(12))
    g1 = scenes.raycast_spheres(cam, centres[:4] + np.array([0.3, 0.2, 2.0]), rng.uniform(0.3, 0.6, 4), 12 + np.arange(4), scale_plane=True)
    keep = g1["depth"] > g0["depth"]
    g1["depth"] = np.where(keep, g1["depth"], 0).astype(f32)
    g1["material_id"] = np.where(keep, g1["material_id"], 0xFFFFFFFF).astype(np.uint32)
    mats = np.concatenate([scenes.hashed_materials(12, 5), scenes.hashed_materials(4, 6, True, (0.2, 0.5))])
    pc = cam.push_constants()
    _, counts, indices = oracle_cluster_lights(oracle, cam, uniforms, lights)
    assert counts.max() > 8
    sc = oracle_scene(pc, uniforms, mats, lights, counts, indices)
    o32, o16 = oracle.shade_opaque_frame(g0, sc)
    levels = oracle.build_pyramid(o16)
    t32, _ = oracle.shade_transmission_frame(g1, sc, levels, ggx_lut, o32, o16)
    with Renderer(w, h, f32_debug=True) as r:
        gpu_setup(r, ggx_lut, uniforms, mats, lights)
        r.build_clusters(cam.write_cluster_data())
        r.assign_lights(cam.assign_lights())
        gc, gi = r.read_cluster_lights(len(counts))
        np.testing.assert_array_equal(gc, counts)
        r.set_gbuffer(0, g0)
        r.set_gbuffer(1, g1)
        r.shade_opaque(pc)
        r.generate_mips()
        r.shade_transmission(pc)
        got = r.read_hdr_f32()
    assert rel_l2(got[..., :3], t32[..., :3]) < REL_L2_TOL


def test_uploads_from_pinned_memory(oracle, ggx_lut):
    """Per-frame uploads from page-locked host memory (asynchronous cudaMemcpyAsync, what bench.py's e2e loop does): the
    frame is the same, bit for bit, as with pageable numpy arrays."""
    import torch
    w, h = 320, 180
    s = scenes.instanced_scene(w, h, n_instances=1500, n_lights=16)
    cam = s["camera"]
    fp = cam.frame_params(host.default_tonemap_params())

    def pinned(a):
        t = torch.empty(max(a.nbytes, 16), dtype=torch.uint8).pin_memory()
        v = t.numpy()[:a.nbytes].view(a.dtype).reshape(a.shape)
        v[...] = a
        return t, v

    with Renderer(w, h) as r:
        _upload_scene(r, ggx_lut, s)
        r.frame(fp)
        ref = r.read_hdr()
        keep_i, inst = pinned(s["instances"])
        keep_l, lights = pinned(s["lights"])
        for _ in range(3):
            r.set_instances(inst)
            r.set_lights(lights)
            r.frame(fp)
        got = r.read_hdr()
        # and the upload really is the data: move everything, render, move back
        moved = inst.copy()
        moved["translation_and_scale"][:, 0] += 0.5
        keep_m, moved_p = pinned(moved)
        r.set_instances(moved_p)
        r.frame(fp)
        other = r.read_hdr()
    assert got.tobytes() == ref.tobytes()
    assert (other != ref).mean() > 0.01
