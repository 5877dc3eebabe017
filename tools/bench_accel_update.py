"""tools/bench_accel_update.py — what the top-level update costs an animated, ray-traced scene: the host update
(tr_update_top_level_acceleration_structure: read back, binned SAH on the host, upload, two synchronisations) against the
device update (tr_update_top_level_acceleration_structure_async: a linear BVH built in stream order).

    python tools/bench_accel_update.py                                  # 4K and 1080p, one context and a 4-context group
    python tools/bench_accel_update.py --sizes 3840x2160 --contexts 1 --seconds 3 --out /tmp/accel_update.json

Scene: config 4 (scenes.instanced_scene: 10k instances, 64 lights), ray queries on, every instance rotated every frame
(a cycle of --cycle precomputed page-locked instance sets, uploaded with tr_set_instances, then the update, then the
frame), as the reference's --rotate-model does.  For every size and layout the two updates alternate, --rounds times
each, on the same contexts.  Per run: host ms inside the update call, host ms to enqueue a frame (upload + update + frame),
wall-clock ms per frame over >= --seconds (ending in a synchronise), device ms of the async build (CUDA events around it on
member 0's stream), the per-pass device totals of member 0 (tr_read_pass_totals) and the SHA-256 of one fixed frame
rendered after the run, which must be the same for both updates.  One JSON line with the card's name and power limit.
Exit status 1 if the hashes differ.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from transmission_renderer_b200 import Renderer, RendererGroup, abi, host, scenes  # noqa: E402


def _lut():
    z = np.load(os.path.join(ROOT, "tests", "golden", "ggx_lut_rg.npz"))
    lut = np.zeros(z["rg"].shape[:2] + (4,), np.uint8)
    lut[..., :2] = z["rg"]
    lut[..., 3] = 255
    return lut


def _upload(r, lut, s):
    r.set_uniforms(s["uniforms"])
    r.set_materials(s["materials"])
    r.set_lights(s["lights"])
    r.set_ggx_lut(lut)
    r.set_instances(s["instances"])
    r.set_primitives(s["primitives"])
    m = s["mesh"]
    r.set_mesh(m["positions"], m["normals"], m["uvs"], m["indices"])
    r.build_clusters(s["camera"].write_cluster_data())


def _quat_mul(a, b):
    x1, y1, z1, w1 = a.T
    x2, y2, z2, w2 = b.T
    return np.stack([w1 * x2 + x1 * w2 + y1 * z2 - z1 * y2, w1 * y2 - x1 * z2 + y1 * w2 + z1 * x2,
                     w1 * z2 + x1 * y2 - y1 * x2 + z1 * w2, w1 * w2 - x1 * x2 - y1 * y2 - z1 * z2], 1)


def _rotated(instances, cycle):
    """`cycle` page-locked instance sets, every instance turned 1 degree more about its own axis in each."""
    import torch
    rng = np.random.default_rng(7)
    axis = rng.normal(size=(len(instances), 3))
    axis /= np.linalg.norm(axis, axis=1, keepdims=True)
    q0 = instances["rotation"].astype(np.float64)
    out = []
    for f in range(cycle):
        a = np.radians(1.0) * (f + 1)
        step = np.concatenate([axis * np.sin(a / 2), np.full((len(axis), 1), np.cos(a / 2))], 1)
        t = torch.empty(len(instances) * abi.instance.itemsize, dtype=torch.uint8).pin_memory()
        inst = t.numpy().view(abi.instance)
        inst[:] = instances
        inst["rotation"] = _quat_mul(step, q0).astype(np.float32)
        out.append((t, inst))
    return out


def _gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout
        return [dict(zip(("index", "name", "power_limit", "sm_max_clock"), (f.strip() for f in l.split(","))))
                for l in out.strip().splitlines()]
    except (OSError, subprocess.SubprocessError):
        return None


def _sha(hdr, srgb):
    return {"hdr_rgba16f": hashlib.sha256(np.ascontiguousarray(hdr).tobytes()).hexdigest(),
            "srgb8": hashlib.sha256(np.ascontiguousarray(srgb).tobytes()).hexdigest()}


def _run(members, group, fp, frames, mode, seconds, torch, stream0):
    """One timed run of `mode` ("host" / "async"); returns its numbers and the hash of a fixed frame rendered after it."""
    update = (lambda r: r.update_top_level_acceleration_structure()) if mode == "host" else \
        (lambda r: r.update_top_level_acceleration_structure_async())

    def frame(k):
        for r in members:
            r.set_instances(frames[k % len(frames)][1])
        t1 = time.perf_counter()
        for r in members:
            update(r)
        t2 = time.perf_counter()
        if group is not None:
            group.frame(fp)
        else:
            members[0].frame(fp)
        return t2 - t1

    def sync():
        if group is not None:
            group.sync()
        else:
            members[0].sync()

    for k in range(len(frames)):   # warm-up: buffers at size, the device builder's primitive table uploaded
        frame(k)
    sync()
    # device time of the update alone (member 0), over a few updates with the stream otherwise idle
    build_ms = []
    for k in range(8):
        members[0].set_instances(frames[k % len(frames)][1])
        b, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        b.record(stream0)
        update(members[0])
        e.record(stream0)
        e.synchronize()
        build_ms.append(b.elapsed_time(e))
    for k in range(len(frames)):
        frame(k)
    sync()
    for r in members:
        r.enable_timing(True)
    n, update_s, enqueue_s = 0, 0.0, 0.0
    t0 = time.perf_counter()
    while True:
        a = time.perf_counter()
        update_s += frame(n)
        enqueue_s += time.perf_counter() - a
        n += 1
        if n >= 20 and time.perf_counter() - t0 >= seconds:
            break
    sync()
    wall = time.perf_counter() - t0
    totals, nt = members[0].pass_totals()
    for r in members:
        r.enable_timing(False)
    frame(0)   # the fixed frame both modes hash
    sync()
    if group is not None:
        sha = _sha(group.read_hdr(), group.read_srgb8())
    else:
        sha = _sha(members[0].read_hdr(), members[0].read_srgb8())
    return {"mode": mode, "frames": n, "wall_s": round(wall, 3), "ms_per_frame": round(wall * 1e3 / n, 4),
            "update_call_ms_per_frame": round(update_s * 1e3 / n, 4), "enqueue_ms_per_frame": round(enqueue_s * 1e3 / n, 4),
            "update_device_ms_member0": {"median": round(float(np.median(build_ms)), 4), "min": round(float(np.min(build_ms)), 4),
                                         "note": "CUDA events around one update call on an idle stream; for the host update this "
                                                 "spans its read-back, host build and upload"},
            "pass_ms_per_frame_member0": {k: round(v / max(nt, 1), 4) for k, v in totals.items()},
            "fixed_frame_sha256": sha}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--sizes", default="3840x2160,1920x1080")
    ap.add_argument("--contexts", default="1,4", help="layouts: 1 = one context, n > 1 = an n-context group on device 0")
    ap.add_argument("--seconds", type=float, default=2.0)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--cycle", type=int, default=8)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if torch.cuda.device_count() == 0:
        sys.exit("bench_accel_update: no CUDA device; this measures the GPU and has no CPU path")
    lut = _lut()
    results = []
    for size in a.sizes.split(","):
        W, H = (int(v) for v in size.split("x"))
        s = scenes.instanced_scene(W, H)
        frames = _rotated(s["instances"], a.cycle)
        n_top = int((s["primitives"]["draw_buffer_index"][s["instances"]["primitive_id"]] < 2).sum())
        for n in (int(v) for v in a.contexts.split(",")):
            members = [Renderer(W, H) for _ in range(n)]
            streams = [torch.cuda.Stream(device=0) for _ in range(n)]
            group = None
            try:
                for r, st in zip(members, streams):
                    r.set_stream(st.cuda_stream)
                    _upload(r, lut, s)
                    r.build_acceleration_structures()
                group = RendererGroup(members) if n > 1 else None
                fp = s["camera"].frame_params(host.default_tonemap_params(), acceleration_structure_address=1)
                if group is None:
                    fp["push_constants"]["acceleration_structure_address"] = members[0].acceleration_structure_address
                runs = []
                for _ in range(a.rounds):
                    for mode in ("host", "async"):
                        runs.append(_run(members, group, fp, frames, mode, a.seconds, torch, streams[0]))
            finally:
                if group is not None:
                    group.close()
                for r in members:
                    r.set_stream(None)
                    r.close()
            hashes = {json.dumps(r["fixed_frame_sha256"], sort_keys=True) for r in runs}
            results.append({"resolution": [W, H], "contexts": n, "top_level_instances": n_top, "runs": runs,
                            "hashes_equal": len(hashes) == 1})
            print(json.dumps(results[-1]), file=sys.stderr)
    result = {"tool": "bench_accel_update", "device": torch.cuda.get_device_name(0), "gpus": _gpu_info(),
              "workload": "config 4: scenes.instanced_scene (10k instances, 64 lights), ray queries on, every instance rotated "
                          "every frame; n > 1 contexts = one tr_group on device 0 (equal bands)",
              "seconds_per_run": a.seconds, "results": results}
    line = json.dumps(result)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")
    return 0 if all(r["hashes_equal"] for r in results) else 1


if __name__ == "__main__":
    sys.exit(main())
