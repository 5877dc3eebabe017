"""Ray-queried shadows with dense cluster lists: up to 128 lights per cluster, so the occluded-ray bits fill all four list
planes of the shadow mask (positions 0-127, `m[i >> 5]` in shadow_mask_kernel, `occluded_word(i)` in shade_kernel), on
every shadowed shading-kernel variant <TRANS, HAS_POS, F32OUT, TEX>, on both light loops (the warp-uniform loop, which
carries most warps of wide frames, and the mixed-warp merge), and on both light tables (shared memory up to 768 lights,
global memory beyond).  The CPU oracle is the reference: masks and G-buffer planes bit for bit, linear HDR within rel-L2
1e-4 and a per-pixel bound, sRGB8 within 2/255.

The scene is shadow_scene with 220 dim point lights appended around the occluders: the six original lights (the
spotlight among them) keep their ids, and 835 of the 320x180 frame's clusters reach the 128-entry clamp.  With that
many dim lights one light more or less moves a pixel by about 1 %, which a frame-level L2 would hide, hence the
per-pixel bound."""
import numpy as np
import pytest

from accel_checks import _upload_scene
from pipeline import REL_L2_TOL, SRGB_TOL, oracle_cluster_lights, oracle_scene, rel_l2
from transmission_renderer_b200 import Renderer, abi, host, scenes

f32 = np.float32
N_DENSE = 220
DENSE_SEED = 0x5EED00B1
DENSE_BOX = ((-4.5, 0.2, -4.5), (4.5, 3.5, 3.0))
MAX_SMEM_LIGHTS = 768          # k_shade.cu: light tables up to this size live in shared memory
SMALL, WIDE = (320, 180), (1920, 1080)
PIXEL_TOL = 1e-3               # per pixel, relative to the pixel's largest channel (+ 1e-3 absolute)


# ---------------------------------------------------------------------------------------------------------- scenes
def _dense_lights(lights):
    """`lights` followed by the dense set, so every original light keeps its id and its place in the lists."""
    return np.concatenate([lights, scenes.hashed_point_lights(N_DENSE, DENSE_SEED, box=DENSE_BOX, intensity=(0.5, 3.0))])


def _scene(kind, w, h):
    s = scenes.shadow_scene(w, h) if kind == "shadow" else scenes.textured_sphere_scene(w, h)
    s["lights"] = _dense_lights(s["lights"])
    return s


def _inert_lights(n):
    """Lights behind the camera, 60-100 m away, with a 0.2 m falloff sphere: they join no cluster, so no list changes."""
    rng = np.random.default_rng(5)
    ls = [host.light_new_point((rng.uniform(-50, 50), rng.uniform(0, 20), rng.uniform(60, 100)), (1.0, 0.8, 0.6), 0.002)
          for _ in range(n)]
    return np.concatenate(ls)


def _with_light_count(lights, n):
    return np.concatenate([lights, _inert_lights(n - len(lights))]) if n > len(lights) else lights


def _positions(g, cam):
    """The G-buffer's world positions decoded in float64, moved 1 cm along the normal (so a kernel that decodes the
    depth instead of reading the plane gets other rays); zero where nothing is covered."""
    h, w = g["depth"].shape
    ys, xs = np.mgrid[0:h, 0:w]
    ndc = np.stack([(xs + 0.5) / w * 2 - 1, (ys + 0.5) / h * 2 - 1, g["depth"].astype(np.float64), np.ones((h, w))], -1)
    q = ndc @ np.linalg.inv(cam.proj_view.astype(np.float64)).T
    n = g["normal"].astype(np.float64)
    n = n / np.maximum(np.linalg.norm(n, axis=-1, keepdims=True), 1e-30)
    pos = q[..., :3] / q[..., 3:] + 0.01 * n
    return np.where((g["depth"] > 0)[..., None], pos, 0.0).astype(f32)


def _cluster_of(g, uniforms):
    """Each pixel's cluster index (-1 where not covered): cluster_index with the column and row in fp32 as the kernels
    compute them, the depth slice restated in float64, so an estimate near slice boundaries."""
    h, w = g["depth"].shape
    u = uniforms[0]
    zn, zf, scale, bias = (float(u[k]) for k in ("z_near", "z_far", "scale", "bias"))
    ys, xs = np.mgrid[0:h, 0:w].astype(f32)
    cx = np.floor((xs + f32(0.5)) / u["cluster_size_in_pixels"][0]).astype(np.int64)
    cy = np.floor((ys + f32(0.5)) / u["cluster_size_in_pixels"][1]).astype(np.int64)
    d = g["depth"].astype(np.float64)
    lin = 2 * zn * zf / (zf + zn - (2 * (1 - d) - 1) * (zf - zn))
    with np.errstate(divide="ignore", invalid="ignore"):
        cz = np.maximum(np.floor(np.log2(lin) * scale + bias), 0).astype(np.int64)
    nx, ny = int(u["num_clusters"][0]), int(u["num_clusters"][1])
    return np.where(d > 0, cz * nx * ny + cy * nx + cx, -1)


def _run_shares(cluster):
    """(runs with a covered pixel, share of them whose covered pixels all sit in one cluster) over the 32-pixel runs of
    the frame in row-major order, the shading kernels' work items."""
    runs = cluster.reshape(-1)
    runs = np.concatenate([runs, np.full(-len(runs) % 32, -1)]).reshape(-1, 32)
    covered = runs >= 0
    lo = np.where(covered, runs, np.iinfo(np.int64).max).min(1)
    hi = runs.max(1)
    some = covered.any(1)
    return int(some.sum()), float((lo[some] == hi[some]).mean())


# ---------------------------------------------------------------------------------------------------------- the oracle
_REFS = {}


def _visibility(oracle, s, textured):
    cam = s["camera"]
    _, visible = oracle.frustum_culling(s["instances"], s["primitives"], cam.culling())
    if textured:
        return oracle.visibility(s["mesh"], s["instances"], s["primitives"], visible, cam.push_constants(), derivatives=True,
                                 materials=s["materials"], textures=s["textures"])
    return oracle.visibility(s["mesh"], s["instances"], s["primitives"], visible, cam.push_constants())


def _shade(oracle, lut, s, g0, g1, shadows=True):
    """Masks, opaque and final HDR and sRGB8 of the G-buffers (g0, g1) on the oracle, with ray queries on."""
    cam = s["camera"]
    _, cc, ci = oracle_cluster_lights(oracle, cam, s["uniforms"], s["lights"])
    sc = oracle_scene(cam.push_constants(), s["uniforms"], s["materials"], s["lights"], cc, ci)
    if "textures" in s:
        sc["textures"] = s["textures"]
    sc["accel"] = oracle.Accel(s["mesh"], s["instances"], s["primitives"]) if shadows else None
    o32, o16 = oracle.shade_opaque_frame(g0, sc)
    t32, t16 = oracle.shade_transmission_frame(g1, sc, oracle.build_pyramid(o16), lut, o32, o16)
    out = dict(g0=g0, g1=g1, counts=cc, indices=ci, o32=o32, o16=o16, t32=t32, t16=t16,
               srgb=oracle.tonemap_frame(t16, host.default_tonemap_params()))
    if shadows:
        out.update(m0=oracle.shadow_mask_frame(g0, sc), m1=oracle.shadow_mask_frame(g1, sc))
    return out


def _reference(oracle, lut, kind, size):
    """The oracle's frame of the dense scene `kind` at `size`, computed once per module."""
    key = (kind, size)
    if key not in _REFS:
        s = _scene(kind, *size)
        g0, g1 = _visibility(oracle, s, kind == "textured")
        _REFS[key] = _shade(oracle, lut, s, g0, g1)
    return _REFS[key]


# ---------------------------------------------------------------------------------------------------------- the GPU
def _gpu_frame(lut, s, f32_debug=True, build="host", unshadowed=False):
    """One tr_frame of `s` with ray queries on; `build`: "host" (tr_build_acceleration_structures) or "device" (the
    stream-ordered build).  `unshadowed` renders the frame once more without the handle."""
    w, h = s["camera"].width, s["camera"].height
    cam = s["camera"]
    params = host.default_tonemap_params()
    with Renderer(w, h, f32_debug=f32_debug) as r:
        if "textures" in s:
            r.set_textures(s["textures"])
        _upload_scene(r, lut, s)
        handle = r.build_acceleration_structures() if build == "host" else r.build_acceleration_structures_async()
        r.frame(cam.frame_params(params, acceleration_structure_address=handle))
        out = dict(m0=r.read_shadow_mask(0), m1=r.read_shadow_mask(1), hdr16=r.read_hdr(), o16=r.read_pyramid_level(0),
                   srgb=r.read_srgb8(), gb0=r.read_gbuffer(0, derivatives="textures" in s),
                   gb1=r.read_gbuffer(1, derivatives="textures" in s))
        if f32_debug:
            out["t32"] = r.read_hdr_f32()
        if unshadowed:
            r.frame(cam.frame_params(params))
            out["lit32"] = r.read_hdr_f32()
    return out


def _off_pixels(got32, ref32):
    """Pixels whose colour is off by more than PIXEL_TOL relative to the reference's largest channel."""
    g, r = got32[..., :3].astype(np.float64), ref32[..., :3].astype(np.float64)
    return np.abs(g - r).max(-1) > PIXEL_TOL * (np.abs(r).max(-1) + 1e-3)


def _check_masks(got, ref):
    for layer in (0, 1):
        a, b = got[f"m{layer}"], ref[f"m{layer}"]
        assert (a != b).sum() == 0, f"layer {layer}: {(a != b).any(0).sum()} pixels' occluded-ray bits differ " \
                                    f"(planes {sorted(set(np.nonzero(a != b)[0].tolist()))})"


def _check_colour(got, ref, what):
    """Opaque fp16 and final fp32 HDR within rel-L2 and the per-pixel bound; sRGB8 within 2/255."""
    e_o = rel_l2(got["o16"].view(np.float16)[..., :3], ref["o16"].view(np.float16)[..., :3])
    e_t = rel_l2(got["t32"][..., :3], ref["t32"][..., :3])
    off = _off_pixels(got["t32"], ref["t32"])
    d = np.abs(got["srgb"].astype(int) - ref["srgb"].astype(int))
    print(f"{what}: opaque fp16 rel-L2 {e_o:.2e}, final fp32 rel-L2 {e_t:.2e}, {off.sum()} pixels off by > {PIXEL_TOL}, "
          f"sRGB8 max diff {d.max()}")
    assert e_o < REL_L2_TOL and e_t < REL_L2_TOL
    assert off.mean() < 1e-4, f"{what}: {off.sum()} pixels off by more than {PIXEL_TOL}"
    assert d.max() <= SRGB_TOL, f"{what}: {(d > SRGB_TOL).sum()} channels off by more than {SRGB_TOL}/255"


def _check_same_bytes(a, b, keys, what):
    for k in keys:
        assert a[k].tobytes() == b[k].tobytes(), f"{what}, {k}: {(a[k] != b[k]).sum()} values differ"


# ---------------------------------------------------------------------------------------------------------- tests
def test_dense_scene_fills_every_list_plane(oracle, ggx_lut):
    """The fixture on the oracle alone (no GPU): some list reaches the 128-entry clamp; both layers have occluded rays
    in every list plane, position 127 among them; the inert lights of the table tests join no cluster; and at the wide
    size most runs with covered pixels sit in one cluster (the warp-uniform loop) while a good share does not, and at
    the small size almost none do (the mixed-warp merge)."""
    ref = _reference(oracle, ggx_lut, "shadow", SMALL)
    assert ref["counts"].max() == abi.TR_MAX_LIGHTS_PER_CLUSTER
    print(f"{(ref['counts'] == abi.TR_MAX_LIGHTS_PER_CLUSTER).sum()} clusters at the clamp")
    for layer in (0, 1):
        m = ref[f"m{layer}"]
        per_plane = [int((m[k] != 0).sum()) for k in range(5)]
        print(f"layer {layer}: pixels with occluded bits per plane (0-3 lists, 4 sun) {per_plane}")
        assert all(n > 0 for n in per_plane[:4]), f"layer {layer}: a list plane is empty"
    assert ((ref["m0"][3] >> 31) & 1).any() or ((ref["m1"][3] >> 31) & 1).any()   # list position 127
    assert (ref["m0"][4] & 1).any()

    s = _scene("shadow", *SMALL)
    cam = s["camera"]
    for n in (MAX_SMEM_LIGHTS, MAX_SMEM_LIGHTS + 1, 1500):
        _, cc, ci = oracle_cluster_lights(oracle, cam, s["uniforms"], _with_light_count(s["lights"], n))
        assert np.array_equal(cc, ref["counts"]) and np.array_equal(ci, ref["indices"]), f"{n} lights change the lists"

    w = _scene("shadow", *WIDE)
    g0, g1 = _visibility(oracle, w, False)
    for layer, g in ((0, g0), (1, g1)):
        n, share = _run_shares(_cluster_of(g, w["uniforms"]))
        print(f"{WIDE[0]}x{WIDE[1]} layer {layer}: {n} runs with covered pixels, {share:.1%} in one cluster")
        if layer == 0:
            assert 0.5 <= share <= 0.9
    n, share = _run_shares(_cluster_of(ref["g0"], s["uniforms"]))
    print(f"{SMALL[0]}x{SMALL[1]} layer 0: {n} runs with covered pixels, {share:.1%} in one cluster")
    assert share < 0.1                                                           # the small frame runs the mixed-warp merge


@pytest.mark.gpu
@pytest.mark.parametrize("size", [SMALL, WIDE], ids=["320x180", "1920x1080"])
def test_dense_lists_frame(oracle, ggx_lut, size):
    """tr_frame with the handle of tr_build_acceleration_structures: 320x180 runs mostly mixed warps, 1920x1080 mostly
    the warp-uniform loop.  Masks bit for bit; the pixels whose occluded lights all sit at list positions >= 32 (so
    only planes 1-3 decide them) each within the per-pixel bound; a context without the fp32 debug target gives the
    same fp16 HDR, opaque mip 0 and sRGB8 bytes."""
    ref = _reference(oracle, ggx_lut, "shadow", size)
    s = _scene("shadow", *size)
    got = _gpu_frame(ggx_lut, s, unshadowed=True)
    for layer in (0, 1):
        for k in ("depth", "normal", "material_id"):
            a, b = got[f"gb{layer}"][k], np.asarray(ref[f"g{layer}"][k]).reshape(got[f"gb{layer}"][k].shape)
            assert a.tobytes() == b.tobytes(), f"layer {layer} plane {k} differs"
    _check_masks(got, ref)
    _check_colour(got, ref, f"dense lists {size[0]}x{size[1]}")

    m0 = ref["m0"]
    high_only = (m0[0] == 0) & (m0[1:4] != 0).any(0) & (ref["g0"]["depth"] > 0) & (ref["g1"]["depth"] == 0)
    off = _off_pixels(got["t32"], ref["t32"])
    lit_off = _off_pixels(got["lit32"], ref["t32"])
    print(f"{high_only.sum()} opaque pixels occluded only at list positions >= 32; the unshadowed frame is off on "
          f"{lit_off[high_only].mean():.1%} of them")
    assert high_only.sum() > 0.005 * size[0] * size[1]
    assert lit_off[high_only].mean() > 0.3                                        # a lost bit shows at the bound
    assert not off[high_only].any(), f"{off[high_only].sum()} pixels occluded only at positions >= 32 are off"

    half = _gpu_frame(ggx_lut, s, f32_debug=False)
    _check_same_bytes(half, got, ("m0", "m1", "hdr16", "o16", "srgb"), "without the fp32 target")


@pytest.mark.gpu
def test_dense_lists_device_built_trees(oracle, ggx_lut):
    """The same frame traced against the trees of tr_build_acceleration_structures_async: masks bit for bit against
    the oracle, and the frame byte-equal to the one traced against the host-built trees."""
    ref = _reference(oracle, ggx_lut, "shadow", SMALL)
    s = _scene("shadow", *SMALL)
    got = _gpu_frame(ggx_lut, s, build="device")
    _check_masks(got, ref)
    _check_same_bytes(got, _gpu_frame(ggx_lut, s), ("t32", "hdr16", "srgb"), "device-built against host-built trees")


@pytest.mark.gpu
def test_light_table_paths(oracle, ggx_lut):
    """Inert lights appended to the dense scene up to exactly 768 lights (the shared-memory table), then 769 and 1 500
    (the global-memory table of the shading kernels).  No list changes and the ids of the real lights stay, so the
    masks, fp16 and fp32 HDR and the opaque mip 0 are byte-equal across the light counts, with and without the handle;
    the frame at the scene's own count is judged against the oracle."""
    ref = _reference(oracle, ggx_lut, "shadow", SMALL)
    s = _scene("shadow", *SMALL)
    cam = s["camera"]
    w, h = SMALL
    params = host.default_tonemap_params()
    runs = {}
    with Renderer(w, h, f32_debug=True) as r:
        _upload_scene(r, ggx_lut, s)
        handle = r.build_acceleration_structures()
        for n in (len(s["lights"]), MAX_SMEM_LIGHTS, MAX_SMEM_LIGHTS + 1, 1500):
            r.set_lights(_with_light_count(s["lights"], n))
            r.frame(cam.frame_params(params, acceleration_structure_address=handle))
            counts, indices = r.read_cluster_lights(len(ref["counts"]))
            assert np.array_equal(counts, ref["counts"]), f"{n} lights: the list lengths changed"
            used = np.arange(abi.TR_MAX_LIGHTS_PER_CLUSTER)[None, :] < counts[:, None]
            assert np.array_equal(indices.reshape(used.shape)[used], ref["indices"].reshape(used.shape)[used]), \
                f"{n} lights: the lists changed"
            shadowed = dict(m0=r.read_shadow_mask(0), m1=r.read_shadow_mask(1), hdr16=r.read_hdr(), t32=r.read_hdr_f32(),
                            o16=r.read_pyramid_level(0), srgb=r.read_srgb8())
            r.frame(cam.frame_params(params))
            lit = dict(hdr16=r.read_hdr(), t32=r.read_hdr_f32(), o16=r.read_pyramid_level(0))
            runs[n] = shadowed, lit
    base = len(s["lights"])
    _check_masks(runs[base][0], ref)
    _check_colour(runs[base][0], ref, f"{base} lights")
    for n in (MAX_SMEM_LIGHTS, MAX_SMEM_LIGHTS + 1, 1500):
        _check_same_bytes(runs[n][0], runs[base][0], ("m0", "m1", "hdr16", "t32", "o16"), f"{n} lights with the handle")
        _check_same_bytes(runs[n][1], runs[base][1], ("hdr16", "t32", "o16"), f"{n} lights without the handle")


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["shadow", "textured"])
def test_position_planes(oracle, ggx_lut, kind):
    """G-buffers with a world-position plane (the HAS_POS kernels, and shadow_mask_kernel<true>): the oracle's planes of
    the dense scene plus positions 1 cm off the surface, uploaded with tr_set_gbuffer and shaded pass by pass with the
    handle.  Masks bit for bit and colours within tolerance against the oracle given the same planes; the mask is not
    the one of the decoded positions, so the plane is what the rays start from.  Without the fp32 target the fp16 HDR,
    opaque mip 0 and sRGB8 bytes are the same."""
    size = SMALL
    base = _reference(oracle, ggx_lut, kind, size)
    s = _scene(kind, *size)
    cam = s["camera"]
    if kind == "textured":
        # with a position plane neither side rebuilds the neighbours' positions from ddepth, so a normal map would get a
        # zero cotangent frame (NaN normals): the normal maps are unbound, every other texture stays
        s["materials"]["textures"][:, scenes.TEX_SLOTS["normal_map"]] = -1
    g0, g1 = (dict(g, position=_positions(g, cam)) for g in (base["g0"], base["g1"]))
    ref = _shade(oracle, ggx_lut, s, g0, g1)
    moved = [(ref[f"m{l}"] != base[f"m{l}"]).any(0).sum() for l in (0, 1)]
    print(f"{kind}: the position plane changes the occluded-ray bits of {moved} pixels")
    assert moved[0] > 50

    def run(f32_debug):
        with Renderer(*size, f32_debug=f32_debug) as r:
            if "textures" in s:
                r.set_textures(s["textures"])
            _upload_scene(r, ggx_lut, s)
            r.assign_lights(cam.assign_lights())
            pc = cam.push_constants(r.build_acceleration_structures())
            r.set_gbuffer(0, g0)
            r.set_gbuffer(1, g1)
            r.shade_opaque(pc)
            out = dict(m0=r.read_shadow_mask(0), o16=r.read_pyramid_level(0))
            r.generate_mips()
            r.shade_transmission(pc)
            r.tonemap(host.default_tonemap_params())
            out.update(m1=r.read_shadow_mask(1), hdr16=r.read_hdr(), srgb=r.read_srgb8())
            if f32_debug:
                out["t32"] = r.read_hdr_f32()
        return out

    got = run(True)
    _check_masks(got, ref)
    _check_colour(got, ref, f"{kind} with position planes")
    _check_same_bytes(run(False), got, ("m0", "m1", "hdr16", "o16", "srgb"), "without the fp32 target")


@pytest.mark.gpu
def test_textured_materials(oracle, ggx_lut):
    """textured_sphere_scene with the dense lights and ray queries on (the TEX kernels, built for two CTAs per SM): masks,
    G-buffer planes and colours against the oracle; without the fp32 target the same fp16 HDR, opaque mip 0 and sRGB8
    bytes."""
    ref = _reference(oracle, ggx_lut, "textured", SMALL)
    s = _scene("textured", *SMALL)
    got = _gpu_frame(ggx_lut, s)
    for layer in (0, 1):
        for k in ("depth", "normal", "uv", "material_id", "duv", "ddepth"):
            a, b = got[f"gb{layer}"][k], np.asarray(ref[f"g{layer}"][k]).reshape(got[f"gb{layer}"][k].shape)
            assert a.tobytes() == b.tobytes(), f"layer {layer} plane {k}: {(a != b).sum()} values differ"
    assert (ref["m0"][:4] != 0).any(0).sum() > 1000 and (ref["m0"][1:4] != 0).any(0).sum() > 100 and (ref["m1"] != 0).any()
    _check_masks(got, ref)
    _check_colour(got, ref, "textured")
    _check_same_bytes(_gpu_frame(ggx_lut, s, f32_debug=False), got, ("m0", "m1", "hdr16", "o16", "srgb"),
                      "without the fp32 target")
