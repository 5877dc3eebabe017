"""tools/bench_accel_build.py — the bottom-level build on the host (tr_build_acceleration_structures: read-back, binned SAH,
upload, three synchronisations) against the device build in stream order (tr_build_acceleration_structures_async).

    python tools/bench_accel_build.py                                     # 1 M and 4 M knot triangles, 4K and 1080p
    python tools/bench_accel_build.py --knot-tris 1048576 --sizes 1920x1080 --seconds 1 --out /tmp/accel_build.json

Scene: config 4 (scenes.instanced_scene: 10k instances, 64 lights) plus one opaque scenes.torus_knot of --knot-tris triangles
that 4 instances share (tools/bench_mesh_update.py).  For every knot size:
  build     one build on an idle stream: GPU ms between CUDA events around the call and wall-clock ms to a synchronise
  reload    tr_set_mesh + build + frame per frame, host build against async build, one context and a 4-context group
  quality   opaque and transmissive pass ms (the shadow rays are traced inside them) of the host tree, the device tree, and
            the host tree refitted from pose 0 to the pose of frame 1, 10 and 100
  rebuild   refit every frame and async rebuild every k frames, wall-clock ms per frame
and the SHA-256 of the frame each variant renders, which must agree.  One JSON line with the card's name and power limit.
Exit status 1 if a pair of hashes differs.
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
from bench_mesh_update import _pinned, _pose, _scene  # noqa: E402
from transmission_renderer_b200 import Renderer, RendererGroup, host  # noqa: E402


def _build(r, mode):
    return r.build_acceleration_structures() if mode == "host" else r.build_acceleration_structures_async()


def _build_times(s, lut, torch, reps):
    out = {}
    st = torch.cuda.Stream(device=0)
    with Renderer(640, 360) as r:
        r.set_stream(st.cuda_stream)
        _upload(r, lut, s)
        for mode in ("host", "async"):
            gpu, wall = [], []
            for k in range(reps + 1):
                r.sync()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                t0 = time.perf_counter()
                e0.record(st)
                _build(r, mode)
                e1.record(st)
                e1.synchronize()
                if k:   # the first build sizes the buffers
                    wall.append((time.perf_counter() - t0) * 1e3)
                    gpu.append(e0.elapsed_time(e1))
            out[mode] = {"gpu_ms_median": round(float(np.median(gpu)), 4), "wall_ms_median": round(float(np.median(wall)), 4),
                         "wall_ms_min": round(float(np.min(wall)), 4)}
        r.set_stream(None)
    return out


def _reload(s, lut, W, H, n, mode, seconds, torch):
    m = s["mesh"]
    members = [Renderer(W, H) for _ in range(n)]
    streams = [torch.cuda.Stream(device=0) for _ in range(n)]
    group = None
    fp = s["camera"].frame_params(host.default_tonemap_params(), acceleration_structure_address=1)
    try:
        for r, st in zip(members, streams):
            r.set_stream(st.cuda_stream)
            _upload(r, lut, s)
        group = RendererGroup(members) if n > 1 else None

        def frame():
            for r in members:
                r.set_mesh(m["positions"], m["normals"], m["uvs"], m["indices"])
                _build(r, mode)
            if group is not None:
                group.frame(fp)
            else:
                fp["push_constants"]["acceleration_structure_address"] = members[0].acceleration_structure_address
                members[0].frame(fp)

        def sync():
            group.sync() if group is not None else members[0].sync()

        frame()   # sizes every buffer
        sync()
        k, t0 = 0, time.perf_counter()
        while k < 1 or time.perf_counter() - t0 < seconds:   # a host reload of millions of triangles takes seconds
            frame()
            k += 1
        sync()
        ms = (time.perf_counter() - t0) * 1e3 / k
        src = group if group is not None else members[0]
        return {"mode": mode, "frames": k, "ms_per_frame": round(ms, 3), "frame_sha256": _sha(src.read_hdr(), src.read_srgb8())}
    finally:
        if group is not None:
            group.close()
        for r in members:
            r.set_stream(None)
            r.close()


def _pass_times(r, fp):
    for _ in range(3):
        r.frame(fp)
    r.sync()
    r.enable_timing(True)
    for _ in range(20):
        r.frame(fp)
    totals, nt = r.pass_totals()
    r.enable_timing(False)
    return {"opaque_ms": round(totals["shade_opaque_ms"] / nt, 4), "transmission_ms": round(totals["shade_transmission_ms"] / nt, 4),
            "frame_sha256": _sha(r.read_hdr(), r.read_srgb8())}


def _quality(s, rng_v, lut, W, H):
    a, b = rng_v
    m = s["mesh"]
    fp = s["camera"].frame_params(host.default_tonemap_params(), acceleration_structure_address=1)
    rows = []
    for f in (1, 10, 100):
        pos = _pose(m["positions"][a:b], m["normals"][a:b], f)
        full = dict(m, positions=m["positions"].copy())
        full["positions"][a:b] = pos
        row = {"frames_of_deformation": f}
        for kind in ("host", "device", "refit"):
            with Renderer(W, H) as r:
                _upload(r, lut, s if kind == "refit" else dict(s, mesh=full))
                _build(r, "async" if kind == "device" else "host")
                if kind == "refit":
                    for g in range(1, f + 1):
                        if g == f or g % 10 == 0:
                            r.update_mesh_vertices(_pose(m["positions"][a:b], m["normals"][a:b], g) if g != f else pos,
                                                   m["normals"][a:b], first_vertex=a)
                    r.update_top_level_acceleration_structure_async()
                fp["push_constants"]["acceleration_structure_address"] = r.acceleration_structure_address
                row[kind] = _pass_times(r, fp)
        row["hashes_equal"] = len({json.dumps(row[k]["frame_sha256"], sort_keys=True) for k in ("host", "device", "refit")}) == 1
        rows.append(row)
        print(json.dumps(row), file=sys.stderr)
    return rows


def _rebuild_every(s, rng_v, lut, W, H, ks, seconds, cycle):
    """Refit every frame (tr_update_mesh_vertices + async top level), async rebuild every k frames instead of the top-level
    update; wall-clock per frame, and the hash of the frame at pose 0 after the run."""
    a, b = rng_v
    m = s["mesh"]
    nrm = m["normals"][a:b]
    poses = [_pinned(_pose(m["positions"][a:b], nrm, f + 1))[1] for f in range(cycle)]
    pose0 = _pinned(_pose(m["positions"][a:b], nrm, 0))[1]
    fp = s["camera"].frame_params(host.default_tonemap_params(), acceleration_structure_address=1)
    out = []
    with Renderer(W, H) as r:
        _upload(r, lut, s)
        fp["push_constants"]["acceleration_structure_address"] = r.build_acceleration_structures_async()
        for k in ks:
            def frame(i):
                r.update_mesh_vertices(poses[i % cycle], nrm, first_vertex=a)
                if k and i % k == k - 1:
                    r.build_acceleration_structures_async()
                else:
                    r.update_top_level_acceleration_structure_async()
                r.frame(fp)
            for i in range(3):
                frame(i)
            r.sync()
            i, t0 = 0, time.perf_counter()
            while i < 3 or time.perf_counter() - t0 < seconds:
                frame(i)
                i += 1
            r.sync()
            ms = (time.perf_counter() - t0) * 1e3 / i
            r.update_mesh_vertices(pose0, nrm, first_vertex=a)
            r.build_acceleration_structures_async()
            r.frame(fp)
            out.append({"rebuild_every": k or None, "frames": i, "ms_per_frame": round(ms, 3),
                        "frame_sha256": _sha(r.read_hdr(), r.read_srgb8())})
            print(json.dumps(out[-1]), file=sys.stderr)
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--knot-tris", default="1048576,4194304")
    ap.add_argument("--sizes", default="3840x2160,1920x1080")
    ap.add_argument("--contexts", default="1,4")
    ap.add_argument("--seconds", type=float, default=1.0)
    ap.add_argument("--build-reps", type=int, default=5)
    ap.add_argument("--rebuild-every", default="0,1,4,16", help="0: never (refit only)")
    ap.add_argument("--quality-size", default="1920x1080")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if torch.cuda.device_count() == 0:
        sys.exit("bench_accel_build: no CUDA device; this measures the GPU and has no CPU path")
    lut = _lut()
    qW, qH = (int(v) for v in a.quality_size.split("x"))
    per_knot = []
    ok = True
    for kt in (int(v) for v in a.knot_tris.split(",")):
        s, rng_v = _scene(qW, qH, kt, 4)
        knot = {"knot_triangles": int(s["primitives"]["index_count"][-1]) // 3, "build": _build_times(s, lut, torch, a.build_reps)}
        print(json.dumps(knot), file=sys.stderr)
        reload = []
        for size in a.sizes.split(","):
            W, H = (int(v) for v in size.split("x"))
            sz, _ = _scene(W, H, kt, 4)
            for n in (int(v) for v in a.contexts.split(",")):
                runs = [_reload(sz, lut, W, H, n, mode, a.seconds, torch) for mode in ("host", "async")]
                eq = runs[0]["frame_sha256"] == runs[1]["frame_sha256"]
                ok = ok and eq
                reload.append({"resolution": [W, H], "contexts": n, "runs": runs, "hashes_equal": eq})
                print(json.dumps(reload[-1]), file=sys.stderr)
        knot["reload"] = reload
        knot["quality"] = _quality(s, rng_v, lut, qW, qH)
        knot["refit_and_rebuild"] = _rebuild_every(s, rng_v, lut, qW, qH, [int(v) for v in a.rebuild_every.split(",")], a.seconds, 4)
        ok = ok and all(q["hashes_equal"] for q in knot["quality"])
        ok = ok and len({json.dumps(x["frame_sha256"], sort_keys=True) for x in knot["refit_and_rebuild"]}) == 1
        per_knot.append(knot)
    result = {"tool": "bench_accel_build", "device": torch.cuda.get_device_name(0), "gpus": _gpu_info(),
              "workload": "config 4 (scenes.instanced_scene: 10k instances, 64 lights) + a torus knot shared by 4 instances; "
                          "n > 1 contexts = one tr_group on device 0 (equal bands)",
              "seconds_per_run": a.seconds, "results": per_knot, "hashes_equal": ok}
    line = json.dumps(result)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
