"""tools/bench_device_animation.py — what a pose computed on the GPU costs a frame when it must go through host memory
(today's path for a host that animates with torch or CUDA) against handing the device array to the library in stream order.

    python tools/bench_device_animation.py                              # 4K and 1080p, ray queries on and off
    python tools/bench_device_animation.py --sizes 1920x1080 --rq off --seconds 1 --out /tmp/device_animation.json

Two workloads, each on one context whose stream is the torch stream that computes the pose (tr_set_stream):
  mesh        config 4 (scenes.instanced_scene: 10k instances, 64 lights) plus the torus knot of tools/bench_mesh_update.py
              (--knot-tris triangles, 4 instances), displaced along its normals every frame by a torch op on the GPU
                host_round_trip  positions and normals copied to page-locked memory, a synchronisation, tr_update_mesh_vertices
                device_source    tr_update_mesh_vertices with the CUDA tensors
  transforms  config 4, every instance rotated about its own axis every frame by a torch op on the GPU (a quaternion product)
                host_round_trip  the (n, 8) transforms copied to page-locked memory, a synchronisation, the records filled on
                                 the host, tr_set_instances
                device_source    tr_update_instance_transforms with the CUDA tensor
With ray queries the update is followed by tr_update_top_level_acceleration_structure_async, then the frame.  Per run:
wall-clock ms per frame over >= --seconds (ending in a synchronise); the device ms of the update alone on an idle stream (CUDA
events around the library call: for the round trip its upload and kernels, plus the device-to-host copy measured the same
way); and the SHA-256 of a fixed frame (one fixed pose) rendered through the run's path, which must be the same for both paths.  One
JSON line with the card's name and power limit.  Exit status 1 if a pair of hashes differs.
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
from bench_mesh_update import AMP, _scene as _knot_scene  # noqa: E402
from transmission_renderer_b200 import Renderer, abi, host, scenes  # noqa: E402


class _Mesh:
    """The knot's pose at frame f, computed on the GPU: p + AMP sin(6x + 4z + 0.05 f) n (tools/bench_mesh_update.py)."""

    def __init__(self, s, rng_v, torch):
        a, b = rng_v
        self.first = a
        self.base_p = torch.from_numpy(s["mesh"]["positions"][a:b].copy()).cuda()
        self.base_n = torch.from_numpy(s["mesh"]["normals"][a:b].copy()).cuda()
        self.pin_p = torch.empty_like(self.base_p, device="cpu").pin_memory()
        self.pin_n = torch.empty_like(self.base_n, device="cpu").pin_memory()
        self.bytes = 2 * self.base_p.numel() * 4

    def pose(self, f):
        x, z = self.base_p[:, 0], self.base_p[:, 2]
        return self.base_p + (AMP * (6.0 * x + 4.0 * z + 0.05 * f).sin())[:, None] * self.base_n, self.base_n

    def to_host(self, dev):
        self.pin_p.copy_(dev[0], non_blocking=True)
        self.pin_n.copy_(dev[1], non_blocking=True)

    def host_update(self, r, stream):
        stream.synchronize()
        r.update_mesh_vertices(self.pin_p.numpy(), self.pin_n.numpy(), first_vertex=self.first)

    def device_update(self, r, dev):
        r.update_mesh_vertices(dev[0], dev[1], first_vertex=self.first)


class _Transforms:
    """Every instance turned 1 degree per frame about its own axis: q(f) = step(f) * q0, as a torch op on the GPU."""

    def __init__(self, s, torch):
        inst = s["instances"]
        rng = np.random.default_rng(7)
        axis = rng.normal(size=(len(inst), 3))
        axis /= np.linalg.norm(axis, axis=1, keepdims=True)
        self.torch = torch
        self.axis = torch.from_numpy(axis.astype(np.float32)).cuda()
        self.ts = torch.from_numpy(np.ascontiguousarray(inst["translation_and_scale"], np.float32)).cuda()
        self.q0 = torch.from_numpy(np.ascontiguousarray(inst["rotation"], np.float32)).cuda()
        self.pin = torch.empty((len(inst), 8), dtype=torch.float32).pin_memory()
        rec = torch.empty(len(inst) * abi.instance.itemsize, dtype=torch.uint8).pin_memory()
        self.keep = rec
        self.records = rec.numpy().view(abi.instance)
        self.records[:] = inst
        self.bytes = len(inst) * 32

    def pose(self, f):
        a = np.radians(1.0) * (f + 1)
        v = self.axis * float(np.sin(a / 2))
        w1 = float(np.cos(a / 2))
        x1, y1, z1 = v[:, 0], v[:, 1], v[:, 2]
        x2, y2, z2, w2 = self.q0.unbind(1)
        q = self.torch.stack([w1 * x2 + x1 * w2 + y1 * z2 - z1 * y2, w1 * y2 - x1 * z2 + y1 * w2 + z1 * x2,
                              w1 * z2 + x1 * y2 - y1 * x2 + z1 * w2, w1 * w2 - x1 * x2 - y1 * y2 - z1 * z2], 1)
        return self.torch.cat([self.ts, q], 1)

    def to_host(self, dev):
        self.pin.copy_(dev, non_blocking=True)

    def host_update(self, r, stream):
        stream.synchronize()
        t = self.pin.numpy()
        self.records["translation_and_scale"] = t[:, :4]
        self.records["rotation"] = t[:, 4:]
        r.set_instances(self.records)

    def device_update(self, r, dev):
        r.update_instance_transforms(dev)


def _run(r, work, path, rq, fp, seconds, torch, stream):
    def update(f):
        with torch.cuda.stream(stream):
            dev = work.pose(f)
            if path == "host_round_trip":
                work.to_host(dev)
                work.host_update(r, stream)
            else:
                work.device_update(r, dev)
        if rq:
            r.update_top_level_acceleration_structure_async()

    def frame(f):
        update(f)
        r.frame(fp)

    for f in range(3):
        frame(f)
    r.sync()
    dev_ms = {}
    for name in ("update", "device_to_host_copy") if path == "host_round_trip" else ("update",):
        ms = []
        for f in range(8):
            with torch.cuda.stream(stream):
                dev = work.pose(f)
            stream.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            with torch.cuda.stream(stream):
                if path == "host_round_trip" and name == "update":   # the pose already in host memory
                    work.to_host(dev)
                    stream.synchronize()
                e0.record(stream)
                if name == "device_to_host_copy":
                    work.to_host(dev)
                elif path == "host_round_trip":
                    work.host_update(r, stream)
                else:
                    work.device_update(r, dev)
                e1.record(stream)
            e1.synchronize()
            ms.append(e0.elapsed_time(e1))
        dev_ms[name] = {"median": round(float(np.median(ms)), 4), "min": round(float(np.min(ms)), 4)}
    if rq:
        r.update_top_level_acceleration_structure_async()
    r.frame(fp)
    r.sync()
    n, t0 = 0, time.perf_counter()
    while True:
        frame(n)
        n += 1
        if n >= 3 and time.perf_counter() - t0 >= seconds:
            break
    r.sync()
    wall = time.perf_counter() - t0
    frame(-1)   # a fixed pose both paths render
    r.sync()
    return {"path": path, "frames": n, "ms_per_frame": round(wall * 1e3 / n, 4), "update_device_ms": dev_ms,
            "fixed_frame_sha256": _sha(r.read_hdr(), r.read_srgb8())}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--sizes", default="3840x2160,1920x1080")
    ap.add_argument("--rq", default="off,on", help="ray queries: on, off or both")
    ap.add_argument("--workloads", default="mesh,transforms")
    ap.add_argument("--knot-tris", type=int, default=1 << 20)
    ap.add_argument("--seconds", type=float, default=1.5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if torch.cuda.device_count() == 0:
        sys.exit("bench_device_animation: no CUDA device; this measures the GPU and has no CPU path")
    lut = _lut()
    results = []
    for size in a.sizes.split(","):
        W, H = (int(v) for v in size.split("x"))
        for wl in a.workloads.split(","):
            if wl == "mesh":
                s, rng_v = _knot_scene(W, H, a.knot_tris, 4)
            else:
                s = scenes.instanced_scene(W, H)
            for rq in (v == "on" for v in a.rq.split(",")):
                stream = torch.cuda.Stream(device=0)
                r = Renderer(W, H)
                try:
                    r.set_stream(stream.cuda_stream)
                    _upload(r, lut, s)
                    handle = r.build_acceleration_structures_async() if rq else 0
                    work = _Mesh(s, rng_v, torch) if wl == "mesh" else _Transforms(s, torch)
                    torch.cuda.synchronize()
                    fp = s["camera"].frame_params(host.default_tonemap_params(), acceleration_structure_address=handle)
                    runs = [_run(r, work, path, rq, fp, a.seconds, torch, stream) for path in ("host_round_trip", "device_source")]
                finally:
                    r.set_stream(None)
                    r.close()
                hashes = {json.dumps(x["fixed_frame_sha256"], sort_keys=True) for x in runs}
                results.append({"workload": wl, "resolution": [W, H], "ray_queries": rq, "source_bytes_per_frame": work.bytes,
                                "runs": runs, "hashes_equal": len(hashes) == 1})
                print(json.dumps(results[-1]), file=sys.stderr)
    knot = int(_knot_scene(64, 64, a.knot_tris, 4)[0]["primitives"]["index_count"][-1]) // 3
    result = {"tool": "bench_device_animation", "device": torch.cuda.get_device_name(0), "gpus": _gpu_info(),
              "workload": f"mesh: config 4 + a torus knot of {knot} triangles (4 instances) displaced every frame on the GPU; "
                          "transforms: config 4 with all 10k instances rotated every frame on the GPU; one context",
              "seconds_per_run": a.seconds, "results": results}
    line = json.dumps(result)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")
    return 0 if all(x["hashes_equal"] for x in results) else 1


if __name__ == "__main__":
    sys.exit(main())
