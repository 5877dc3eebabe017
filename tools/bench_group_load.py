"""tools/bench_group_load.py — load-to-first-frame of a tr_group: every member loaded on its own (the uploads, image binds and
structure builds repeated per member) against one member loaded and the scene copied to the others GPU to GPU
(tr_group_replicate_scene).

    python tools/bench_group_load.py                                  # 4 contexts on device 0; all devices when there are 2+
    python tools/bench_group_load.py --images 8 --size 1920x1080 --reps 1 --out /tmp/group_load.json

Scene: config 4 (scenes.instanced_scene: 10k instances, 64 lights) plus a 1 048 576-triangle torus knot shared by 4 instances
(tools/bench_mesh_update.py), and --images sRGB images of --image-side² bound with tr_set_texture_async from pageable level 0
(8 distinct images, bound in turn), the diffuse image of opaque material k being image k mod --images.  The acceleration
structures are built with tr_build_acceleration_structures_async, and the frame traces shadow rays against them.

Every timed run starts from freshly created contexts and a fresh group (their creation is not timed) and ends when the
first group frame has been read back.  Reported per member set (one device, several devices):
  per_member   wall-clock ms from the first upload to the first frame read back, every member loaded
  replicate    the same with member 0 loaded and tr_group_replicate_scene, plus the call's GPU time (CUDA events on member
               0's stream around the call: from the point the load had reached to the end of every copy) and its
               host time; and, after the frame, one more replicate on idle streams (GPU ms)
and the SHA-256 of the first frame of every run, which must all agree.  One JSON line with the cards' names and power
limits.  Exit status 1 if two hashes differ.
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
from bench_mesh_update import _scene  # noqa: E402
from transmission_renderer_b200 import Renderer, RendererGroup, host, scenes  # noqa: E402


def _textured(s, n_images):
    mats = s["materials"].copy()
    opaque = np.nonzero(mats["transmission_factor"] == 0)[0]
    for j, m in enumerate(opaque):
        mats["textures"][m, scenes.TEX_SLOTS["diffuse"]] = j % n_images
    return dict(s, materials=mats)


def _load(r, lut, s, images):
    for i in range(len(images[1])):
        r.set_texture_async(i, images[0][images[1][i]], True)
    _upload(r, lut, s)
    return r.build_acceleration_structures_async()


def _run(route, devices, W, H, lut, s, images, torch):
    members = [Renderer(W, H, device=d) for d in devices]
    streams = [torch.cuda.Stream(device=d) for d in devices]
    group = None
    try:
        for r, st in zip(members, streams):
            r.set_stream(st.cuda_stream)
        group = RendererGroup(members)
        for d in set(devices):
            torch.cuda.synchronize(d)
        out = {"route": route}
        t0 = time.perf_counter()
        if route == "per_member":
            for r in members:
                _load(r, lut, s, images)
        else:
            _load(members[0], lut, s, images)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(streams[0])
            t1 = time.perf_counter()
            group.replicate_scene(0)
            out["replicate_host_ms"] = round((time.perf_counter() - t1) * 1e3, 3)
            e1.record(streams[0])
        fp = s["camera"].frame_params(host.default_tonemap_params(), acceleration_structure_address=1)
        group.frame(fp)   # each member's own handle (RendererGroup.frame)
        srgb = group.read_srgb8()
        out["load_to_first_frame_ms"] = round((time.perf_counter() - t0) * 1e3, 2)
        out["frame_sha256"] = _sha(group.read_hdr(), srgb)
        if route == "replicate":
            out["replicate_gpu_ms"] = round(e0.elapsed_time(e1), 3)
            group.sync()
            e0.record(streams[0])
            group.replicate_scene(0)
            e1.record(streams[0])
            e1.synchronize()
            out["replicate_idle_gpu_ms"] = round(e0.elapsed_time(e1), 3)
        return out
    finally:
        if group is not None:
            group.close()
        for r in members:
            r.set_stream(None)
            r.close()


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--size", default="3840x2160")
    ap.add_argument("--knot-tris", type=int, default=1048576)
    ap.add_argument("--images", type=int, default=64)
    ap.add_argument("--image-side", type=int, default=2048)
    ap.add_argument("--contexts", type=int, default=4, help="members on device 0")
    ap.add_argument("--reps", type=int, default=2, help="runs of each route, alternating")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    n_dev = torch.cuda.device_count()
    if n_dev == 0:
        sys.exit("bench_group_load: no CUDA device; this measures the GPU and has no CPU path")
    W, H = (int(v) for v in a.size.split("x"))
    lut = _lut()
    s, _ = _scene(W, H, a.knot_tris, 4)
    s = _textured(s, a.images)
    rng = np.random.default_rng(9)
    distinct = [rng.integers(0, 256, (a.image_side, a.image_side, 4), dtype=np.uint8) for _ in range(min(8, a.images))]
    images = (distinct, [i % len(distinct) for i in range(a.images)])
    sets = [[0] * a.contexts]
    if n_dev >= 2:
        sets.append(list(range(min(8, n_dev))))
    _run("replicate", sets[0][:2], W, H, lut, s, images, torch)   # warm-up: modules, allocator pools
    results, hashes = [], set()
    for devices in sets:
        runs = []
        for _ in range(a.reps):
            for route in ("per_member", "replicate"):
                runs.append(_run(route, devices, W, H, lut, s, images, torch))
                hashes.add(json.dumps(runs[-1]["frame_sha256"], sort_keys=True))
                print(json.dumps({"devices": devices, **runs[-1]}), file=sys.stderr)
        results.append({"devices": devices, "runs": runs})
    ok = len(hashes) == 1
    result = {"tool": "bench_group_load", "device": torch.cuda.get_device_name(0), "gpus": _gpu_info(), "resolution": [W, H],
              "workload": f"config 4 (10k instances, 64 lights) + a {int(s['primitives']['index_count'][-1]) // 3}-triangle torus "
                          f"knot shared by 4 instances, {a.images} sRGB {a.image_side}x{a.image_side} images bound with "
                          "tr_set_texture_async from pageable level 0, tr_build_acceleration_structures_async, shadow rays on",
              "results": results, "hashes_equal": ok}
    line = json.dumps(result)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
