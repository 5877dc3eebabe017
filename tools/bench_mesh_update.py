"""tools/bench_mesh_update.py — what vertex animation costs a frame: a full reload (tr_set_mesh, plus
tr_build_acceleration_structures with ray queries: host chunk spheres and host bottom-level build, each with a
synchronisation) against tr_update_mesh_vertices (the changed vertices in stream order, chunk spheres and a bottom-level refit
on the device, plus the async top-level update with ray queries).

    python tools/bench_mesh_update.py                                  # 4K and 1080p, ray queries on and off, 1 and 4 contexts
    python tools/bench_mesh_update.py --sizes 1920x1080 --contexts 1 --rq on --seconds 1 --out /tmp/mesh_update.json

Scene: config 4 (scenes.instanced_scene: 10k instances, 64 lights) plus one opaque scenes.torus_knot of --knot-tris triangles
(default about 1 M) that --knot-instances instances share.  Every frame displaces the knot along its normals by a moving sine (a
cycle of --cycle precomputed poses, page-locked).  For every size, ray-query setting and layout the two modes alternate on the
same contexts:
  reload  tr_set_mesh with the whole mesh (+ tr_build_acceleration_structures) + frame
  update  tr_update_mesh_vertices with the knot's vertices (+ tr_update_top_level_acceleration_structure_async) + frame
Per run: wall-clock ms per frame (ending in a synchronise), device ms of one update of member 0 on an idle stream (CUDA events:
the whole call, and a one-vertex call, which runs the same kernels over the whole mesh with a 12-byte copy), and the SHA-256
of a fixed frame rendered after the run, which must be the same for both modes.  Then the drift of a refitted tree: the
opaque + transmissive pass times (they contain the shadow-ray pass) of a context refitted from pose 0 to the pose of frame
1, 10 and 100, against a context freshly built at that pose, and the hashes of both frames.  One JSON line with the card's
name and power limit.  Exit status 1 if a pair of hashes differs.
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from bench_accel_update import _gpu_info, _lut, _sha, _upload  # noqa: E402
from transmission_renderer_b200 import Renderer, RendererGroup, abi, host, scenes  # noqa: E402

AMP = 0.05   # displacement amplitude, in the knot's object units (the knot is about 1.7 across)


def _scene(W, H, knot_tris, knot_instances):
    """config 4 + one large shared torus knot; returns the scene and the knot's vertex range."""
    s = scenes.instanced_scene(W, H)
    n_v = 128
    n_u = max(8, int(round(knot_tris / (2 * n_v))))
    pos, nrm, uv, idx = scenes.torus_knot(n_u=n_u, n_v=n_v)
    m = s["mesh"]
    v0, i0 = len(m["positions"]), len(m["indices"])
    mesh = dict(positions=np.concatenate([m["positions"], pos]), normals=np.concatenate([m["normals"], nrm]),
                uvs=np.concatenate([m["uvs"], uv]), indices=np.concatenate([m["indices"], idx + np.uint32(v0)]))
    p = np.zeros(1, abi.primitive_info)
    lo, hi = pos.min(0), pos.max(0)
    # the caller's bounding sphere must hold every pose: the static one, widened by the displacement amplitude
    p["packed_bounding_sphere"][0] = (*((lo + hi) / 2), np.linalg.norm((hi - lo).astype(np.float64)) / 2 + AMP)
    p["index_count"] = len(idx)
    p["first_index"] = i0
    p["first_instance"] = len(s["primitives"])
    prim = len(s["primitives"])
    inst = [scenes.make_instance((-12.0 + 8.0 * k, 3.0, -6.0 - 3.0 * (k % 2)), 3.0, (0.0, 0.0, 0.0, 1.0), prim, k % len(s["materials"]))
            for k in range(knot_instances)]
    return dict(s, mesh=mesh, primitives=np.concatenate([s["primitives"], p]),
                instances=np.concatenate([s["instances"]] + inst)), (v0, v0 + len(pos))


def _pose(base_pos, base_nrm, f):
    """The knot at frame f: displaced along its normals by a sine moving 0.05 rad per frame."""
    p = base_pos.astype(np.float64)
    a = AMP * np.sin(6.0 * p[:, 0] + 4.0 * p[:, 2] + 0.05 * f)
    return (p + a[:, None] * base_nrm).astype(np.float32)


def _pinned(a):
    import torch
    t = torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    return t, t.numpy()


def _run(members, group, fp, s, rng_v, poses, mode, rq, seconds, torch, stream0):
    a, b = rng_v
    m = s["mesh"]
    knot_nrm = m["normals"][a:b]
    full = dict(m)

    def sync():
        group.sync() if group is not None else members[0].sync()

    def frame(k):
        pin = poses[k % len(poses)]
        for r in members:
            if mode == "reload":
                full["positions"] = pin[2]
                r.set_mesh(full["positions"], full["normals"], full["uvs"], full["indices"])
                if rq:
                    r.build_acceleration_structures()
            else:
                r.update_mesh_vertices(pin[1], knot_nrm, first_vertex=a)
                if rq:
                    r.update_top_level_acceleration_structure_async()
        if group is not None:
            group.frame(fp)
        else:
            if rq:
                fp["push_constants"]["acceleration_structure_address"] = members[0].acceleration_structure_address
            members[0].frame(fp)

    for k in range(2):
        frame(k)
    sync()
    dev = {}
    if mode == "update":   # device time of the update alone (member 0, idle stream)
        for name, n in (("whole_call", b - a), ("kernels_one_vertex_call", 1)):
            ms = []
            for k in range(8):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream0)
                members[0].update_mesh_vertices(poses[k % len(poses)][1][:n], knot_nrm[:n], first_vertex=a)
                if rq:
                    members[0].update_top_level_acceleration_structure_async()
                e1.record(stream0)
                e1.synchronize()
                ms.append(e0.elapsed_time(e1))
            dev[name] = {"median": round(float(np.median(ms)), 4), "min": round(float(np.min(ms)), 4)}
        frame(0)
        sync()
    n, t0 = 0, time.perf_counter()
    while True:
        frame(n)
        n += 1
        if n >= 3 and time.perf_counter() - t0 >= seconds:
            break
    sync()
    wall = time.perf_counter() - t0
    frame(0)   # the fixed frame both modes hash
    sync()
    src = group if group is not None else members[0]
    return {"mode": mode, "frames": n, "ms_per_frame": round(wall * 1e3 / n, 4),
            "update_device_ms_member0": dev or None, "fixed_frame_sha256": _sha(src.read_hdr(), src.read_srgb8())}


def _drift(s, rng_v, lut, W, H, torch):
    """Opaque + transmissive pass ms (shadow rays included) of a tree refitted from pose 0 against a fresh one."""
    a, b = rng_v
    m = s["mesh"]
    out = []
    fp = s["camera"].frame_params(host.default_tonemap_params(), acceleration_structure_address=1)
    for f in (1, 10, 100):
        pos = _pose(m["positions"][a:b], m["normals"][a:b], f)
        full = dict(m, positions=m["positions"].copy())
        full["positions"][a:b] = pos
        row = {"frames_of_deformation": f}
        for kind in ("refit", "fresh"):
            with Renderer(W, H) as r:
                _upload(r, lut, s if kind == "refit" else dict(s, mesh=full))
                r.build_acceleration_structures()
                if kind == "refit":
                    for g in range(1, f + 1):   # poses on the way (every tenth), as an animation would
                        if g == f or g % 10 == 0:
                            r.update_mesh_vertices(_pose(m["positions"][a:b], m["normals"][a:b], g) if g != f else pos,
                                                   m["normals"][a:b], first_vertex=a)
                    r.update_top_level_acceleration_structure_async()
                fp["push_constants"]["acceleration_structure_address"] = r.acceleration_structure_address
                for _ in range(3):
                    r.frame(fp)
                r.sync()
                r.enable_timing(True)
                for _ in range(20):
                    r.frame(fp)
                totals, nt = r.pass_totals()
                r.enable_timing(False)
                row[kind] = {"opaque_ms": round(totals["shade_opaque_ms"] / nt, 4),
                             "transmission_ms": round(totals["shade_transmission_ms"] / nt, 4),
                             "frame_sha256": _sha(r.read_hdr(), r.read_srgb8())}
        row["hashes_equal"] = row["refit"]["frame_sha256"] == row["fresh"]["frame_sha256"]
        out.append(row)
        print(json.dumps(row), file=sys.stderr)
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--sizes", default="3840x2160,1920x1080")
    ap.add_argument("--contexts", default="1,4", help="layouts: 1 = one context, n > 1 = an n-context group on device 0")
    ap.add_argument("--rq", default="on,off", help="ray queries: on, off or both")
    ap.add_argument("--knot-tris", type=int, default=1 << 20)
    ap.add_argument("--knot-instances", type=int, default=4)
    ap.add_argument("--seconds", type=float, default=1.5)
    ap.add_argument("--cycle", type=int, default=4)
    ap.add_argument("--drift-size", default="1920x1080")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if torch.cuda.device_count() == 0:
        sys.exit("bench_mesh_update: no CUDA device; this measures the GPU and has no CPU path")
    lut = _lut()
    results = []
    for size in a.sizes.split(","):
        W, H = (int(v) for v in size.split("x"))
        s, rng_v = _scene(W, H, a.knot_tris, a.knot_instances)
        lo, hi = rng_v
        poses = []
        for f in range(a.cycle):
            pos = _pose(s["mesh"]["positions"][lo:hi], s["mesh"]["normals"][lo:hi], f + 1)
            full = s["mesh"]["positions"].copy()
            full[lo:hi] = pos
            t, pin = _pinned(pos)
            poses.append((t, pin, full))
        for rq in (v == "on" for v in a.rq.split(",")):
            for n in (int(v) for v in a.contexts.split(",")):
                members = [Renderer(W, H) for _ in range(n)]
                streams = [torch.cuda.Stream(device=0) for _ in range(n)]
                group = None
                try:
                    for r, st in zip(members, streams):
                        r.set_stream(st.cuda_stream)
                        _upload(r, lut, s)
                        if rq:
                            r.build_acceleration_structures()
                    group = RendererGroup(members) if n > 1 else None
                    fp = s["camera"].frame_params(host.default_tonemap_params(), acceleration_structure_address=1 if rq else 0)
                    runs = [_run(members, group, fp, s, rng_v, poses, mode, rq, a.seconds, torch, streams[0])
                            for mode in ("reload", "update")]
                finally:
                    if group is not None:
                        group.close()
                    for r in members:
                        r.set_stream(None)
                        r.close()
                hashes = {json.dumps(r["fixed_frame_sha256"], sort_keys=True) for r in runs}
                results.append({"resolution": [W, H], "ray_queries": rq, "contexts": n, "runs": runs, "hashes_equal": len(hashes) == 1})
                print(json.dumps(results[-1]), file=sys.stderr)
    W, H = (int(v) for v in a.drift_size.split("x"))
    s, rng_v = _scene(W, H, a.knot_tris, a.knot_instances)
    drift = _drift(s, rng_v, lut, W, H, torch)
    knot_tris = int(s["primitives"]["index_count"][-1]) // 3
    result = {"tool": "bench_mesh_update", "device": torch.cuda.get_device_name(0), "gpus": _gpu_info(),
              "workload": f"config 4 (scenes.instanced_scene: 10k instances, 64 lights) + a torus knot of {knot_tris} triangles "
                          f"shared by {a.knot_instances} instances, displaced along its normals every frame; n > 1 contexts = "
                          "one tr_group on device 0 (equal bands)",
              "seconds_per_run": a.seconds, "results": results, "refit_drift": {"resolution": [W, H], "poses": drift}}
    line = json.dumps(result)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")
    ok = all(r["hashes_equal"] for r in results) and all(d["hashes_equal"] for d in drift)
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
