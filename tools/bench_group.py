"""tools/bench_group.py — the 4K config-4 frame (scenes.instanced_scene(3840, 2160)) through single-process groups (tr_group_*).

    python tools/bench_group.py --contexts 4 --devices 0,0,0,0      # 4 bands on one GPU: what the group path costs
    python tools/bench_group.py --contexts 8                        # 8 bands over the visible devices
    python tools/bench_group.py --groups 4 --contexts 2             # config 5's 4 x 2 layout: 4 views, 2 bands each

G groups of N contexts each; group g renders orbit view g (yaw 360 g / 64, as config 5's views).  --devices lists the device of
every context, group by group (G * N entries); by default the contexts are spread over the visible devices in contiguous
blocks.  After --warmup group frames, --steps (>= 20) frames of every group are timed with CUDA events on every member's
stream and with a host clock that ends in tr_group_sync.  One JSON line: device names and power limits, the layout, ms per
frame and Mpx/s, every member's per-pass device time, and per group the SHA-256 of the stitched RGBA16F and sRGB8 frame next
to that of one context rendering the same frame in the same run.  Writes nothing unless --out is given.  Exit status 1 if a
group's frame differs from the single context's.
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
from transmission_renderer_b200 import Renderer, RendererGroup, host, scenes  # noqa: E402


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


def _sha(hdr, srgb):
    return {"hdr_rgba16f": hashlib.sha256(np.ascontiguousarray(hdr).tobytes()).hexdigest(),
            "srgb8": hashlib.sha256(np.ascontiguousarray(srgb).tobytes()).hexdigest()}


def _gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout
        return [dict(zip(("index", "name", "power_limit", "sm_max_clock"), (f.strip() for f in l.split(","))))
                for l in out.strip().splitlines()]
    except (OSError, subprocess.SubprocessError):
        return None


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--contexts", type=int, default=2, help="members per group (bands of one frame)")
    ap.add_argument("--groups", type=int, default=1, help="independent groups, each rendering its own orbit view")
    ap.add_argument("--devices", default=None, help="comma-separated device of every context, group by group")
    ap.add_argument("--width", type=int, default=3840)
    ap.add_argument("--height", type=int, default=2160)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = ap.parse_args()
    if a.steps < 20:
        ap.error("--steps: at least 20 timed frames")
    import torch
    n_dev = torch.cuda.device_count()
    if n_dev == 0:
        sys.exit("bench_group: no CUDA device; this measures the GPU and has no CPU path")
    G, N, W, H = a.groups, a.contexts, a.width, a.height
    total = G * N
    devices = [int(d) for d in a.devices.split(",")] if a.devices else [i * n_dev // total for i in range(total)]
    if len(devices) != total:
        ap.error(f"--devices names {len(devices)} devices for {G} groups of {N} contexts")

    lut = _lut()
    s = scenes.instanced_scene(W, H)
    yaws = [360.0 * g / 64 for g in range(G)]
    params = [scenes.Camera(W, H, (0.0, 6.0, 0.0), y, -10.0).frame_params(host.default_tonemap_params()) for y in yaws]

    members = [Renderer(W, H, device=d) for d in devices]
    streams = [torch.cuda.Stream(device=d) for d in devices]
    groups = []
    try:
        for r, st in zip(members, streams):
            _upload(r, lut, s)
            r.set_stream(st.cuda_stream)   # the timing events below go on the members' own streams
        groups = [RendererGroup(members[g * N:(g + 1) * N]) for g in range(G)]
        for _ in range(a.warmup):
            for g, p in zip(groups, params):
                g.frame(p)
        for g in groups:
            g.sync()
        for r in members:
            r.enable_timing(True)
        begin, end = [], []
        for d, st in zip(devices, streams):
            with torch.cuda.device(d):
                e = torch.cuda.Event(enable_timing=True)
                e.record(st)
                begin.append(e)
        t0 = time.perf_counter()
        for _ in range(a.steps):
            for g, p in zip(groups, params):
                g.frame(p)
        for d, st in zip(devices, streams):
            with torch.cuda.device(d):
                e = torch.cuda.Event(enable_timing=True)
                e.record(st)
                end.append(e)
        for g in groups:
            g.sync()
        host_ms = (time.perf_counter() - t0) * 1e3 / a.steps
        event_ms = max(b.elapsed_time(e) for b, e in zip(begin, end)) / a.steps
        per_member = []
        for k, r in enumerate(members):
            totals, n = r.pass_totals()
            r.enable_timing(False)
            g = groups[k // N]
            per_member.append({"group": k // N, "member": k % N, "device": devices[k],
                               "rows": [g.bounds[k % N], g.bounds[k % N + 1]], "frames": n,
                               "pass_ms_per_frame": {key: round(v / max(n, 1), 4) for key, v in totals.items()}})
        hashes = []
        for gi, (g, p) in enumerate(zip(groups, params)):
            got = _sha(g.read_hdr(), g.read_srgb8())
            with Renderer(W, H, device=devices[gi * N]) as one:
                _upload(one, lut, s)
                one.frame(p)
                want = _sha(one.read_hdr(), one.read_srgb8())
            hashes.append({"group": gi, "yaw_deg": yaws[gi], "group_frame": got, "single_context": want, "equal": got == want})
    finally:
        for g in groups:
            g.close()
        for r in members:
            r.set_stream(None)
            r.close()

    used = sorted(set(devices))
    result = {
        "tool": "bench_group",
        "devices": {str(d): torch.cuda.get_device_name(d) for d in used},
        "gpus": _gpu_info(),
        "layout": {"groups": G, "contexts_per_group": N, "device_of_each_context": devices,
                   "contexts_per_device": {str(d): devices.count(d) for d in used}},
        "resolution": [W, H],
        "workload": "config 4: scenes.instanced_scene (10k instances, 64 lights, 30 % transmissive); group g = orbit view g of 64",
        "steps": a.steps, "warmup": a.warmup,
        "ms_per_frame": round(host_ms, 4),
        "ms_per_frame_events": round(event_ms, 4),
        "mpx_per_s": round(G * W * H / (host_ms * 1e-3) / 1e6, 2),
        "members": per_member,
        "frame_sha256": hashes,
    }
    line = json.dumps(result)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")
    return 0 if all(h["equal"] for h in hashes) else 1


if __name__ == "__main__":
    sys.exit(main())
