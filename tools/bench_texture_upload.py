"""tools/bench_texture_upload.py — what binding a glTF scene's images costs, and what rebinding one costs a stream of frames:

    (a) scenes.make_mips on the host + tr_set_texture (the Python ingest today);
    (b) tr_set_texture with the chains already built (the library's share of (a));
    (c) tr_set_texture_async from page-locked level-0 arrays (the chain built on the device).

    python tools/bench_texture_upload.py                         # 64 sRGB images of 2048x2048, 4K frames
    python tools/bench_texture_upload.py --images 8 --size 1024 --frame 1920x1080 --out /tmp/tex.json

Scene: scenes.textured_sphere_scene at the frame size, its materials sampling images 0-7 of --images bound ones.  Per path,
on a fresh context with everything but the images uploaded: wall-clock ms from the first bind to the first frame read back.
Then the device time of the chain kernels for one image (torch.profiler, kernels texture_level0_kernel /
texture_level_kernel), the bytes they move (level 0: 4 B in + 16 B out per texel; level k: 16 + 4 + 16 B), the bandwidth
that is, and tr_measure_hbm_copy beside it.  Streaming: --stream-frames frames enqueued back to back, image 0 rebound before
each one (two alternating sources), blocking call against async call, against the same frames without rebinds.  Every path
must render the same frame (SHA-256 of the sRGB8 and RGBA16F frames); exit status 1 if not.  One JSON line with the card's
name and power limit.
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
from transmission_renderer_b200 import Renderer, host, scenes  # noqa: E402


def _lut():
    z = np.load(os.path.join(ROOT, "tests", "golden", "ggx_lut_rg.npz"))
    lut = np.zeros(z["rg"].shape[:2] + (4,), np.uint8)
    lut[..., :2] = z["rg"]
    lut[..., 3] = 255
    return lut


def _gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout
        return [dict(zip(("index", "name", "power_limit", "sm_max_clock"), (f.strip() for f in l.split(","))))
                for l in out.strip().splitlines()]
    except (OSError, subprocess.SubprocessError):
        return None


def _sha(r):
    return hashlib.sha256(r.read_srgb8().tobytes() + r.read_hdr().tobytes()).hexdigest()


def _images(n, size, base):
    """n sRGB images: the scene's eight procedural ones tiled up to `size`, then seeded noise over a gradient."""
    out = []
    for i in range(n):
        if i < len(base):
            src = base[i]["levels"][0]
            img = np.tile(src, (size // src.shape[0] + 1, size // src.shape[1] + 1, 1))[:size, :size].copy()
        else:
            rng = np.random.default_rng(1000 + i)
            g = (np.arange(size) * 255 // max(size - 1, 1)).astype(np.uint8)
            img = rng.integers(0, 64, (size, size, 4), dtype=np.uint8) + (g[None, :, None] // 2 + g[:, None, None] // 4)
        out.append(np.ascontiguousarray(img, np.uint8))
    return out


def _pinned(a):
    import torch
    t = torch.empty(a.nbytes, dtype=torch.uint8).pin_memory()
    v = t.numpy().reshape(a.shape)
    v[...] = a
    return t, v


def _context(s, lut):
    w, h = s["camera"].width, s["camera"].height
    r = Renderer(w, h)
    r.set_uniforms(s["uniforms"])
    r.set_materials(s["materials"])
    r.set_lights(s["lights"])
    r.set_ggx_lut(lut)
    r.set_instances(s["instances"])
    r.set_primitives(s["primitives"])
    m = s["mesh"]
    r.set_mesh(m["positions"], m["normals"], m["uvs"], m["indices"])
    r.build_clusters(s["camera"].write_cluster_data())
    r.sync()
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=64)
    ap.add_argument("--size", type=int, default=2048)
    ap.add_argument("--frame", default="3840x2160")
    ap.add_argument("--stream-frames", type=int, default=60)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    w, h = (int(v) for v in a.frame.split("x"))
    lut = _lut()
    s = scenes.textured_sphere_scene(w, h)
    imgs = _images(a.images, a.size, s["textures"])
    fp = s["camera"].frame_params(host.default_tonemap_params())
    res = dict(gpu=_gpu_info(), images=a.images, size=a.size, frame=[w, h])

    # ---- (a) make_mips on the host + tr_set_texture
    r = _context(s, lut)
    t0 = time.perf_counter()
    chains = []
    for i, img in enumerate(imgs):
        chains.append(scenes.make_mips(img, True))
        r.set_texture(i, chains[-1], True)
    r.frame(fp)
    r.sync()
    res["load_ms_make_mips_blocking"] = (time.perf_counter() - t0) * 1e3
    hashes = {"make_mips_blocking": _sha(r)}
    r.close()
    # ---- (b) tr_set_texture with the chains built
    r = _context(s, lut)
    t0 = time.perf_counter()
    for i, c in enumerate(chains):
        r.set_texture(i, c, True)
    r.frame(fp)
    r.sync()
    res["load_ms_blocking_prebuilt"] = (time.perf_counter() - t0) * 1e3
    hashes["blocking_prebuilt"] = _sha(r)
    r.close()
    # ---- (c) tr_set_texture_async from page-locked level 0
    pins = [_pinned(img) for img in imgs]
    r = _context(s, lut)
    t0 = time.perf_counter()
    for i, (_, p) in enumerate(pins):
        r.set_texture_async(i, p, True)
    r.frame(fp)
    r.sync()
    res["load_ms_async"] = (time.perf_counter() - t0) * 1e3
    hashes["async"] = _sha(r)

    # ---- device time of the chain kernels, one image, rebinding index 0 in place
    for _ in range(3):
        r.set_texture_async(0, pins[0][1], True)
    r.sync()
    reps = 20
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            r.set_texture_async(0, pins[0][1], True)
        r.sync()
    kern = {}
    for e in prof.events():
        if "texture_level" in e.name and e.device_type.name == "CUDA":
            key = "level0" if "level0" in e.name else "levels"
            kern[key] = kern.get(key, 0.0) + e.time_range.elapsed_us() / 1e3   # us -> ms
    n_lv = host.mip_levels_for_size(a.size, a.size)
    texels = [max(1, a.size >> k) ** 2 for k in range(n_lv)]
    bytes_alg = 20 * texels[0] + 36 * sum(texels[1:])
    kms = {k: v / reps for k, v in kern.items()}
    res["chain_kernels"] = dict(launches_per_image=n_lv, ms_level0=kms.get("level0"), ms_levels_1_on=kms.get("levels"),
                                ms_total=sum(kms.values()), algorithmic_bytes=bytes_alg,
                                gb_per_s=bytes_alg / (sum(kms.values()) * 1e-3) / 1e9 if kms else None,
                                level0_gb_per_s=20 * texels[0] / (kms["level0"] * 1e-3) / 1e9 if "level0" in kms else None,
                                note="working set of one image (84 MB at level 0) fits the 126 MB L2; level 0's bytes were just "
                                     "copied in")
    res["hbm_copy_gb_per_s"] = r.measure_hbm_copy()
    r.sync()

    # ---- streaming: image 0 rebound before every frame, frames back to back
    alt = [pins[0][1], pins[1][1]]
    alt_chains = [chains[0], chains[1]]
    stream = {}
    for mode in ("none", "blocking", "async", "none", "blocking", "async"):
        for k in range(2):            # warm-up
            r.set_texture_async(0, alt[k], True)
            r.frame(fp)
        r.sync()
        t0 = time.perf_counter()
        for f in range(a.stream_frames):
            if mode == "blocking":
                r.set_texture(0, alt_chains[f % 2], True)
            elif mode == "async":
                r.set_texture_async(0, alt[f % 2], True)
            r.frame(fp)
        r.sync()
        ms = (time.perf_counter() - t0) * 1e3 / a.stream_frames
        stream.setdefault(mode, []).append(ms)
        if mode != "none":
            hashes[f"stream_{mode}"] = _sha(r)   # image 1 last (an even frame count) or image 0
    res["stream_ms_per_frame"] = stream
    r.set_texture(0, chains[0], True)
    r.frame(fp)
    r.sync()
    hashes["after_streaming_blocking_image0"] = _sha(r)
    r.close()
    res["hashes"] = hashes
    load = {hashes[k] for k in ("make_mips_blocking", "blocking_prebuilt", "async", "after_streaming_blocking_image0")}
    res["hashes_equal"] = len(load) == 1 and hashes["stream_blocking"] == hashes["stream_async"]
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")
    return 0 if res["hashes_equal"] else 1


if __name__ == "__main__":
    sys.exit(main())
