"""Ray-queried shadows (`--ray-tracing`: src/main.rs:577-658, src/acceleration_structures.rs, shader/src/lighting.rs:97-125)
through the C ABI against the CPU oracle: ray batches and the per-pixel occluded-ray bits bit for bit, frames within the
HDR tolerance, the call-order rules of the handle."""
import numpy as np
import pytest

from accel_checks import _random_rays, _reference, _surface_rays, _upload_scene
from pipeline import REL_L2_TOL, rel_l2
from transmission_renderer_b200 import Renderer, TrError, abi, host, scenes

pytestmark = pytest.mark.gpu
f32 = np.float32


@pytest.mark.parametrize("kind", ["shadow", "instanced"])
def test_ray_batches_bit_exact(oracle, ggx_lut, kind):
    """trace_shadow_ray for random rays (axis-parallel and -0 components included) and for rays cast the way the shaders
    cast them; the product's binned-SAH trees against the oracle's median-split trees and its tree-less definition."""
    w, h = 320, 180
    s = scenes.shadow_scene(w, h) if kind == "shadow" else scenes.instanced_scene(w, h, n_instances=2000, n_lights=16)
    acc = oracle.Accel(s["mesh"], s["instances"], s["primitives"])
    rng = np.random.default_rng(17)
    box = ([-8, 0, -10], [8, 6, 6]) if kind == "shadow" else ([-30, 0, -30], [30, 12, 30])
    o, d, t = _random_rays(rng, 200000, *box)
    po, pd, pt = _surface_rays(s, oracle, 100000, rng)
    with Renderer(w, h) as r:
        _upload_scene(r, ggx_lut, s)
        with pytest.raises(TrError):
            r.trace_shadow_rays(o[:4], d[:4], t[:4])                                  # nothing built yet
        handle = r.build_acceleration_structures()
        assert handle != 0
        got, got_p = r.trace_shadow_rays(o, d, t), r.trace_shadow_rays(po, pd, pt)
    ref, ref_p = acc.trace(o, d, t), acc.trace(po, pd, pt)
    assert (got != ref).sum() == 0 and (got_p != ref_p).sum() == 0
    assert 0.02 < 1 - ref.mean() < 0.98 and 0.02 < 1 - ref_p.mean() < 0.98
    sub = slice(0, 20000)
    assert np.array_equal(got[sub], acc.trace(o[sub], d[sub], t[sub], brute=True))


@pytest.mark.parametrize("size", [(640, 360), (333, 187)])
def test_shadowed_frame(oracle, ggx_lut, size):
    """Whole frames with the handle in PushConstants.acceleration_structure_address: the occluded-ray bits of both layers
    bit for bit (sun + one ray per clustered light, lighting.rs:22-32, 64-71, 154-165, 186-195), linear HDR within 1e-4."""
    w, h = size
    s = scenes.shadow_scene(w, h)
    cam = s["camera"]
    acc = oracle.Accel(s["mesh"], s["instances"], s["primitives"])
    ref = _reference(oracle, ggx_lut, s, acc)
    lit = _reference(oracle, ggx_lut, s, None)
    with Renderer(w, h, f32_debug=True) as r:
        _upload_scene(r, ggx_lut, s)
        handle = r.build_acceleration_structures()
        r.frame(cam.frame_params(host.default_tonemap_params(), acceleration_structure_address=handle))
        m0, m1 = r.read_shadow_mask(0), r.read_shadow_mask(1)
        got32 = r.read_hdr_f32()
        got_o16 = r.read_pyramid_level(0)
        # the same context without the handle renders the unshadowed frame
        r.frame(cam.frame_params(host.default_tonemap_params()))
        got_lit = r.read_hdr_f32()
    ref_m0, ref_m1 = oracle.shadow_mask_frame(ref["g0"], ref["scene"]), oracle.shadow_mask_frame(ref["g1"], ref["scene"])
    assert (m0 != ref_m0).sum() == 0, f"opaque layer: {(m0 != ref_m0).any(0).sum()} pixels differ"
    assert (m1 != ref_m1).sum() == 0, f"transmissive layer: {(m1 != ref_m1).any(0).sum()} pixels differ"
    assert (ref_m0[4] & 1).sum() > 100 and (ref_m0[:4] != 0).any(0).sum() > 1000 and (ref_m1 != 0).any(0).sum() > 50
    e_o = rel_l2(oracle.f16_to_f32(got_o16)[..., :3], oracle.f16_to_f32(ref["o16"])[..., :3])
    e_t = rel_l2(got32[..., :3], ref["t32"][..., :3])
    e_lit = rel_l2(got_lit[..., :3], lit["t32"][..., :3])
    print(f"shadowed {w}x{h}: opaque fp16 rel-L2 {e_o:.2e}, final fp32 rel-L2 {e_t:.2e}; without the handle {e_lit:.2e}")
    assert e_o < REL_L2_TOL and e_t < REL_L2_TOL and e_lit < REL_L2_TOL
    # the L2 norm of this scene is carried by a few very bright pixels next to the low light, so also per pixel:
    off = np.abs(got32[..., :3] - ref["t32"][..., :3]).max(-1) > 1e-3 * (np.abs(ref["t32"][..., :3]).max(-1) + 1e-3)
    assert off.mean() < 1e-4, f"{off.sum()} pixels off by more than 1e-3"
    changed = np.abs(got_lit[..., :3] - ref["t32"][..., :3]).sum(-1) > 0.05 * ref["t32"][..., :3].sum(-1)
    assert changed.mean() > 0.05                                                 # the shadows matter


def test_instanced_scene_shadows(oracle, ggx_lut):
    """Thousands of rotated, scaled instances of eight primitives (two-level traversal under load), 32 lights."""
    w, h = 400, 225
    s = scenes.instanced_scene(w, h, n_instances=3000, n_lights=32)
    cam = s["camera"]
    acc = oracle.Accel(s["mesh"], s["instances"], s["primitives"])
    ref = _reference(oracle, ggx_lut, s, acc)
    with Renderer(w, h, f32_debug=True) as r:
        _upload_scene(r, ggx_lut, s)
        handle = r.build_acceleration_structures()
        r.frame(cam.frame_params(host.default_tonemap_params(), acceleration_structure_address=handle))
        m0, m1 = r.read_shadow_mask(0), r.read_shadow_mask(1)
        got32 = r.read_hdr_f32()
    assert (m0 != oracle.shadow_mask_frame(ref["g0"], ref["scene"])).sum() == 0
    assert (m1 != oracle.shadow_mask_frame(ref["g1"], ref["scene"])).sum() == 0
    e_t = rel_l2(got32[..., :3], ref["t32"][..., :3])
    print(f"instanced shadows {w}x{h}: final fp32 rel-L2 {e_t:.2e}")
    assert e_t < REL_L2_TOL


def test_handle_rules(oracle, ggx_lut):
    """A foreign handle is refused; moving an instance needs the top-level update (src/main.rs:1263-1345) and the update
    is what the next frame traces against; rebinding the mesh invalidates everything."""
    w, h = 320, 180
    s = scenes.shadow_scene(w, h)
    cam = s["camera"]
    with Renderer(w, h, f32_debug=True) as r:
        _upload_scene(r, ggx_lut, s)
        with pytest.raises(TrError) as e:
            r.frame(cam.frame_params(acceleration_structure_address=0x1234))
        assert e.value.status == -1
        handle = r.build_acceleration_structures()
        with pytest.raises(TrError):
            r.frame(cam.frame_params(acceleration_structure_address=handle + 64))
        r.frame(cam.frame_params(acceleration_structure_address=handle))
        before = r.read_shadow_mask(0)
        moved = s["instances"].copy()
        moved["translation_and_scale"][1, :3] += (1.5, 0.4, 0.5)                 # the big sphere
        r.set_instances(moved)
        with pytest.raises(TrError) as e:
            r.frame(cam.frame_params(acceleration_structure_address=handle))
        assert e.value.status == -6
        handle = r.update_top_level_acceleration_structure()
        r.frame(cam.frame_params(acceleration_structure_address=handle))
        after = r.read_shadow_mask(0)
        got32 = r.read_hdr_f32()
        m = s["mesh"]
        r.set_mesh(m["positions"], m["normals"], m["uvs"], m["indices"])
        with pytest.raises(TrError):
            r.frame(cam.frame_params(acceleration_structure_address=handle))
    assert (before != after).any(0).mean() > 0.01
    s2 = dict(s, instances=moved)
    ref = _reference(oracle, ggx_lut, s2, oracle.Accel(s2["mesh"], s2["instances"], s2["primitives"]))
    assert (after != oracle.shadow_mask_frame(ref["g0"], ref["scene"])).sum() == 0
    assert rel_l2(got32[..., :3], ref["t32"][..., :3]) < REL_L2_TOL


def test_band_contexts_trace_their_rows(oracle, ggx_lut):
    """A band context (multi-GPU sharding, DESIGN.md section 5) traces and shades only its rows; the rows equal the
    whole-frame context's rows bit for bit."""
    w, h = 320, 180
    s = scenes.shadow_scene(w, h)
    cam = s["camera"]
    with Renderer(w, h, f32_debug=True) as r:
        _upload_scene(r, ggx_lut, s)
        handle = r.build_acceleration_structures()
        r.frame(cam.frame_params(acceleration_structure_address=handle))
        full_mask, full = r.read_shadow_mask(0), r.read_pyramid_level(0)
    y0, y1 = 60, 120
    with Renderer(w, h, f32_debug=True, band=(y0, y1)) as r:
        _upload_scene(r, ggx_lut, s)
        handle = r.build_acceleration_structures()
        r.frame(cam.frame_params(acceleration_structure_address=handle))
        band_mask, band = r.read_shadow_mask(0), r.read_pyramid_level(0)   # the opaque result (no band exchange here)
    assert np.array_equal(band_mask[:, y0:y1], full_mask[:, y0:y1]) and np.array_equal(band[y0:y1], full[y0:y1])
