"""Helpers shared by the acceleration-structure and ray-query tests: scene upload, rays, the oracle's reference frame,
structure checks of the top and bottom levels, page-locked copies, a held-up stream, and the library's constants.  torch is
imported inside the functions that need it, so the modules that import these collect without a GPU."""
import numpy as np

from pipeline import gpu_setup, oracle_cluster_lights, oracle_scene

f32 = np.float32
ACCEL_STACK = 64               # kAccelStack, tr_device_accel.cuh
ASYNC_TLAS_LAUNCHES = 19       # kAsyncTlasLaunches: count, scan, records, bounds, codes, 4 x (histogram, scan, scatter), hierarchy, boxes
MESH_UPDATE_LAUNCHES = 3       # chunk spheres; with built acceleration structures also the refit's gather and boxes
MESH_UPDATE_LAUNCHES_NO_ACCEL = 1


# ---------------------------------------------------------------------------------------------------------- scenes and rays
def _upload_scene(r, lut, s):
    gpu_setup(r, lut, s["uniforms"], s["materials"], s["lights"])
    r.set_instances(s["instances"])
    r.set_primitives(s["primitives"])
    m = s["mesh"]
    r.set_mesh(m["positions"], m["normals"], m["uvs"], m["indices"])
    r.build_clusters(s["camera"].write_cluster_data())


def _random_rays(rng, n, lo, hi):
    o = rng.uniform(lo, hi, (n, 3)).astype(f32)
    d = rng.normal(size=(n, 3))
    d = (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(f32)
    d[::7, rng.integers(0, 3)] = 0.0
    d[::11] = np.sign(d[::11]) * (np.abs(d[::11]) > 0.5)
    t = rng.uniform(0.5, 60, n).astype(f32)
    ok = np.linalg.norm(d, axis=1) > 0
    return o[ok], d[ok], t[ok]


def _surface_rays(s, oracle, n, rng):
    """Rays as the shaders cast them: from points on the visible surfaces towards the lights and the sun."""
    cam = s["camera"]
    _, visible = oracle.frustum_culling(s["instances"], s["primitives"], cam.culling())
    g0, _ = oracle.visibility(s["mesh"], s["instances"], s["primitives"], visible, cam.push_constants())
    ys, xs = np.nonzero(g0["depth"] > 0)
    pick = rng.choice(len(ys), n)
    ys, xs = ys[pick], xs[pick]
    inv = np.linalg.inv(cam.proj_view.astype(np.float64))
    ndc = np.stack([(xs + 0.5) / cam.width * 2 - 1, (ys + 0.5) / cam.height * 2 - 1, g0["depth"][ys, xs], np.ones(n)], 1)
    h = ndc @ inv.T
    pos = (h[:, :3] / h[:, 3:]).astype(f32)
    lp = s["lights"]["position_and_spotlight_epsilon"][rng.integers(0, len(s["lights"]), n), :3]
    vec = lp - pos
    dist = np.linalg.norm(vec, axis=1).astype(f32)
    return pos, (vec / dist[:, None]).astype(f32), dist


def _reference(oracle, lut, s, accel):
    cam = s["camera"]
    pc = cam.push_constants()
    _, visible = oracle.frustum_culling(s["instances"], s["primitives"], cam.culling())
    g0, g1 = oracle.visibility(s["mesh"], s["instances"], s["primitives"], visible, pc)
    _, cc, ci = oracle_cluster_lights(oracle, cam, s["uniforms"], s["lights"])
    sc = oracle_scene(pc, s["uniforms"], s["materials"], s["lights"], cc, ci)
    sc["accel"] = accel
    o32, o16 = oracle.shade_opaque_frame(g0, sc)
    levels = oracle.build_pyramid(o16)
    t32, t16 = oracle.shade_transmission_frame(g1, sc, levels, lut, o32, o16)
    return dict(g0=g0, g1=g1, scene=sc, o32=o32, o16=o16, t32=t32)


def _deform(mesh, k, first=0, last=None, amp=0.04):
    """Vertices [first, last) displaced along their normals by a moving sine, normals tilted with it: (positions, normals)
    of the range and the whole new mesh."""
    last = len(mesh["positions"]) if last is None else last
    p = mesh["positions"][first:last].astype(np.float64)
    n = mesh["normals"][first:last].astype(np.float64)
    a = amp * np.sin(3.0 * p[:, 0] + 2.0 * p[:, 2] + 0.9 * k)
    newp = (p + a[:, None] * n).astype(f32)
    newn = n + 0.2 * np.cos(2.0 * p[:, 1] + 0.7 * k)[:, None] * np.array([0.3, 0.0, -0.2])
    newn = (newn / np.linalg.norm(newn, axis=1, keepdims=True)).astype(f32)
    full = dict(mesh)
    full["positions"] = mesh["positions"].copy()
    full["normals"] = mesh["normals"].copy()
    full["positions"][first:last] = newp
    full["normals"][first:last] = newn
    return newp, newn, full


# ---------------------------------------------------------------------------------------------------------- structures
def _tree_checks(nodes, inst):
    """Every leaf once, every inner box the exact union of its subtree; returns the depth (inner nodes on the longest path)."""
    m = len(inst)
    if m == 0:
        assert len(nodes) == 1 and nodes["c0"][0] == -1 and nodes["c1"][0] == -1
        assert np.all(np.isinf(nodes["lo0"])) and np.all(np.isinf(nodes["lo1"]))
        return 1
    seen = np.zeros(m, np.int64)
    depth = 0

    def box_of(c):   # (lo, hi) of a child reference
        if c < 0:
            code = ~int(c) & 0xFFFFFFFF
            first, count = code & 0x0FFFFFFF, (code >> 28) + 1
            seen[first:first + count] += 1
            return inst["lo"][first:first + count].min(0), inst["hi"][first:first + count].max(0)
        return walk(c)

    stack_boxes = {}

    def walk(root):   # iterative post-order: (node, depth, children done)
        nonlocal depth
        todo = [(root, 1, False)]
        while todo:
            n, d, done = todo.pop()
            depth = max(depth, d)
            kids = [int(nodes["c0"][n]), int(nodes["c1"][n])]
            if m == 1 and n == 0:
                kids = kids[:1]
            if not done:
                todo.append((n, d, True))
                for c in kids:
                    if c >= 0:
                        todo.append((c, d + 1, False))
                continue
            lo, hi = [], []
            for k, c in enumerate(kids):
                b = stack_boxes.pop(c) if c >= 0 else box_of(c)
                want_lo, want_hi = nodes["lo0" if k == 0 else "lo1"][n], nodes["hi0" if k == 0 else "hi1"][n]
                assert np.array_equal(want_lo, b[0]) and np.array_equal(want_hi, b[1]), \
                    f"node {n} child {k}: box is not the union of its subtree"
                lo.append(b[0])
                hi.append(b[1])
            stack_boxes[n] = (np.min(lo, 0), np.max(hi, 0))
        return stack_boxes.pop(root)

    walk(0)
    if m == 1:
        assert np.all(np.isinf(nodes["lo1"][0])) and np.all(np.isinf(nodes["hi1"][0]))
    assert (seen == 1).all(), "a top-level instance is missing or repeated"
    return depth


def _blas_layout(nodes, prims):
    """(root node, first triangle) of every primitive: the trees lie one after the other in preorder."""
    roots, bases, root, base = [], [], 0, 0
    for p in prims:
        roots.append(root)
        bases.append(base)
        base += int(p["index_count"]) // 3
        todo, count = [root], 0
        while todo:
            n = todo.pop()
            count += 1
            for c in (int(nodes["c0"][n]), int(nodes["c1"][n])):
                if c >= 0:
                    todo.append(c)
        root += count
    assert root == len(nodes)
    return roots, bases


def _check_blas(nodes, tris, prims, mesh):
    """Per primitive: the triangles are the mesh's, as a multiset; every box is the exact union of its subtree (a zero may
    carry either sign)."""
    pos, idx = mesh["positions"], mesh["indices"]
    roots, bases = _blas_layout(nodes, prims)
    inf = np.float32(np.inf)
    for p, (root, base) in enumerate(zip(roots, bases)):
        nt = int(prims["index_count"][p]) // 3
        want = pos[idx[int(prims["first_index"][p]):int(prims["first_index"][p]) + nt * 3]].reshape(nt, 9)
        got = tris[base:base + nt, :, :3].reshape(nt, 9)
        assert (tris[base:base + nt, :, 3] == 0).all()
        key = lambda a: np.sort(np.ascontiguousarray(a + f32(0)).view(np.dtype((np.void, 36))).reshape(-1))
        assert key(got).tobytes() == key(want).tobytes(), f"primitive {p}: triangles differ"
        end = roots[p + 1] if p + 1 < len(roots) else len(nodes)
        boxes = {}

        def leaf(c):
            code = ~c & 0xFFFFFFFF
            first, count = code & 0x0FFFFFFF, (code >> 28) + 1
            t = tris[base + first:base + first + count, :, :3].reshape(-1, 3)
            return t.min(0), t.max(0)

        for n in range(end - 1, root - 1, -1):   # children after their parent
            c0, c1 = int(nodes["c0"][n]), int(nodes["c1"][n])
            if c0 == c1:                           # the special roots
                assert n == root
                assert np.all(nodes["lo1"][n] == inf) and np.all(nodes["hi1"][n] == -inf)
                if nt == 0:
                    assert np.all(nodes["lo0"][n] == inf) and np.all(nodes["hi0"][n] == -inf)
                else:
                    lo, hi = leaf(c0)
                    assert np.array_equal(nodes["lo0"][n], lo) and np.array_equal(nodes["hi0"][n], hi)
                continue
            los, his = [], []
            for k, c in enumerate((c0, c1)):
                lo, hi = leaf(c) if c < 0 else boxes.pop(c)
                assert np.array_equal(nodes["lo0" if k == 0 else "lo1"][n], lo), f"primitive {p} node {n} child {k}"
                assert np.array_equal(nodes["hi0" if k == 0 else "hi1"][n], hi), f"primitive {p} node {n} child {k}"
                los.append(lo)
                his.append(hi)
            boxes[n] = np.min(los, 0), np.max(his, 0)


def _records_key(inst):
    """Top-level records as a multiset, blas_root left out (a fresh build makes other trees), +0 for -0."""
    rec = inst.copy()
    for f in ("translation", "inv_scale", "conj_rotation", "lo", "hi"):
        rec[f] = rec[f] + f32(0)
    rec["blas_root"] = 0
    return np.sort(np.frombuffer(rec.tobytes(), np.dtype((np.void, 64))))


# ---------------------------------------------------------------------------------------------------------- streams
def _pinned(a):
    """A page-locked copy of `a`, structured or not: (the pinned uint8 tensor, which keeps the memory alive, and the copy, a
    view of it with the array's dtype and shape)."""
    import torch
    a = np.ascontiguousarray(a)
    t = torch.empty(a.nbytes, dtype=torch.uint8).pin_memory()
    out = t.numpy().view(a.dtype).reshape(a.shape)
    out[...] = a
    return t, out


def _hold(stream, seconds):
    import torch
    clock_khz = getattr(torch.cuda.get_device_properties(0), "clock_rate", 0) or 2_100_000
    with torch.cuda.stream(stream):
        torch.cuda._sleep(int(seconds * clock_khz * 1e3))   # >= `seconds`: the cycles at the highest clock
