#!/usr/bin/env python
"""bench.py — the headline benchmark of the B200-native light-transport path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference]
                    [--workload 4k|config1|config2|config3|config5|1080p|8k] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

Metric (BASELINE.json): shaded Mpixels/s (opaque + transmission) at 4K; one "step" is one frame of the
record() sequence (src/main.rs:1551-2263) through libtr.so: frustum cull -> light assignment -> visibility
-> opaque shading -> [opaque-band exchange] -> mip chain -> transmissive shading -> tonemap.  Workload =
BASELINE.json configs[3]: 3840x2160, 10 000 instances, 64 point lights, ~97 % opaque and ~97 % frosted-
glass coverage (scenes.instanced_scene).  N > 1 shards the frame into horizontal bands (strong scaling:
the frame is fixed), with the opaque bands exchanged before the mip chain.

`value`  whole-job Mpx/s with every input resident in HBM.
`e2e`    the same frames through the public API with HOST buffers: per step the instances, lights and
         frame constants go host->device from pinned memory and the tonemapped sRGB8 band comes back.
`--workload`  4k = BASELINE.json configs[3] (the headline, default); config1/2/3/5 = configs[0]/[1]/[2]/[4] at their
         stated sizes (config5: 8K x 64 orbit views; combine with --view-groups for the 8x1/4x2/2x4/1x8 sweep).
`--steps K`  the number of timed steps of `value` (and of `e2e`, timed separately through host buffers).
`sustained`  with --min-seconds S > 0: the same frames back to back for >= S seconds with its own clock summary, next to
         the K-step burst (off by default, so that K alone sets how many steps are timed).
`--dump-outputs DIR`  after the timed steps, the frame their last step produced, as a caller of tr_frame receives it:
         DIR/hdr_rgba.npy (the RGBA16F HDR frame, overflows to inf written as the largest finite half, 65504) and
         DIR/srgb8_rgba.npy (the tonemapped sRGB8 frame), both widened to float32, of the whole frame (N > 1: stitched from the bands; with several views a step, view groups or
         --emulate-band: rank 0's rows of the last frame it rendered; --impl reference: the rows of its band).  A frame
         larger than the 64 MB budget is sampled: DUMP_PIXELS pixels chosen by a fixed seed, so that the same arguments
         give the same pixels.
`frame_sha256`  SHA-256 of the whole HDR (RGBA16F) and sRGB8 frame, at N > 1 stitched from the ranks' bands: equal at every N
         <=> N-GPU output == 1-GPU output bitwise, checkable from the JSON lines alone.  `band_hashes` are the per-band
         digests (the N = 1 line carries those of the equal-row splits into 2, 4 and 8); `band_rows` the boundaries used —
         at N > 1 they are balanced by measured cost before the timed region (--equal-bands keeps tr_comm_init's).
`--impl reference`  the reference's per-pixel code (shader + glam-pbr) as the CPU oracle port, all host
         threads (OpenMP), on a bounded band of the same 4K frame.  The reference is Rust -> SPIR-V and
         cannot be built here (no cargo/rustc), so the port under oracle/ is the only runnable form.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    "4k": dict(kind="instanced", width=3840, height=2160, n_instances=10000, n_lights=64,
               name="configs[3]: 4K frosted glass, 10k instances, 64 lights"),
    "1080p": dict(kind="instanced", width=1920, height=1080, n_instances=10000, n_lights=64, name="config-4 scene at 1080p"),
    "8k": dict(kind="instanced", width=7680, height=4320, n_instances=10000, n_lights=64, name="configs[4] scene at 8K, one view"),
    "config1": dict(kind="config1", width=512, height=512, n_instances=0, n_lights=0,
                    name="configs[0]: 512x512 synthetic G-buffer, 1 directional light, roughness 0.25 (mips -> fragment_transmission -> tonemap)"),
    "config2": dict(kind="spheres", knot=False, width=1920, height=1080, n_instances=65, n_lights=4,
                    name="configs[1]: 1080p opaque only, 64 UV-spheres, 4 point lights"),
    "config3": dict(kind="spheres", knot=True, width=1920, height=1080, n_instances=66, n_lights=4,
                    name="configs[2]: 1080p rough transmissive displaced torus knot: opaque -> mip chain -> transmission"),
    "config5": dict(kind="instanced", width=7680, height=4320, n_instances=10000, n_lights=64, views=64,
                    name="configs[4]: 8K, 64 camera views"),
}
HBM_FALLBACK_GBS = 6650.0  # /opt/skills/guides/B200_PROFILING.md fallback


def load_lut():
    z = np.load(os.path.join(ROOT, "tests", "golden", "ggx_lut_rg.npz"))
    lut = np.zeros(z["rg"].shape[:2] + (4,), np.uint8)
    lut[..., :2] = z["rg"]
    lut[..., 3] = 255
    return lut


def make_scene(wl):
    from transmission_renderer_b200 import scenes
    if wl["kind"] == "instanced":
        return scenes.instanced_scene(wl["width"], wl["height"], n_instances=wl["n_instances"], n_lights=wl["n_lights"])
    if wl["kind"] == "spheres":
        return scenes.sphere_grid_scene(wl["width"], wl["height"], transmissive_knot=wl["knot"])
    if wl["kind"] == "config1":
        return scenes.config1(wl["width"], 0.25)
    raise ValueError(wl["kind"])


def base_config(wl, args, world):
    """`config` of the JSON line — the same dict (keys and values) from the B200 arm and from --impl reference."""
    groups = max(1, min(args.view_groups, world))
    bands = world // groups
    return {"workload": wl["name"], "width": wl["width"], "height": wl["height"], "instances": wl["n_instances"],
            "lights": wl["n_lights"], "views": args.views, "parallelism": f"bands{bands}" + (f"xviews{groups}" if groups > 1 else ""),
            "exchange": args.exchange if bands > 1 else "none", "ray_queries": bool(args.ray_tracing),
            "l2": "GPU arm: inputs larger than L2 — the G-buffer, visibility and frame planes touched per frame "
                  f"(~{110 * wl['width'] * wl['height'] / 1e6:.0f} MB) against 126 MB of L2" if wl["width"] * wl["height"] >= 1920 * 1080 else
                  "GPU arm: the working set (~29 MB) fits L2; a 256 MB buffer is overwritten between timed steps (L2 flush)"}


def ncu_traffic(kernel, workload, world):
    """(DRAM bytes per launch of `kernel`, source) from the newest committed `ncu --set full` capture of this workload /
    GPU count — NOT measured in this run (ncu replays kernels; a bench number is never taken under it)."""
    for name in ("r02_dram_traffic.json", "r01_dram_traffic.json"):
        try:
            d = json.load(open(os.path.join(ROOT, "profiles", name)))
            if d.get("workload") == workload and d.get("n_gpus") == world and kernel in d["bytes_per_launch"]:
                return d["bytes_per_launch"][kernel], f"committed capture profiles/{name} (not measured in this run)"
        except Exception:
            pass
    return None, None


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return float(d["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs"
        except Exception:
            pass
    return HBM_FALLBACK_GBS, "fallback (B200_PROFILING.md)"


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    """nvidia-smi clocks + throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows = []
        self.proc = None
        self.gpu = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except subprocess.TimeoutExpired:
                self.proc.kill()

    def summary(self, t0=None, t1=None):
        sm, smax, power, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for t, line in self.rows:
            if t0 is not None and not (t0 - 0.05 <= t <= t1 + 0.15):
                continue
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax.append(float(f[2]))
                power.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(smax)), "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": float(max(power))}


# ----------------------------------------------------------------------------- algorithmic work (SURVEY.md 8d, Appendix C)
def pixel_light_counts(uniforms, depth, cluster_counts, y0, y1):
    """L per pixel = cluster_light_counts[cluster(px)] (shader/src/lib.rs:205-215, shared-structs:54-63)."""
    f32 = np.float32
    u = uniforms[0]
    h, w = depth.shape
    ys, xs = np.mgrid[y0:y1, 0:w]
    d = depth[y0:y1]
    cx = ((xs + f32(0.5)) / f32(u["cluster_size_in_pixels"][0])).astype(np.int64)
    cy = ((ys + f32(0.5)) / f32(u["cluster_size_in_pixels"][1])).astype(np.int64)
    zn, zf = f32(u["z_near"]), f32(u["z_far"])
    rng = f32(2) * (f32(1) - d) - f32(1)
    with np.errstate(divide="ignore", invalid="ignore"):
        lin = (f32(2) * zn * zf) / (zf + zn - rng * (zf - zn))
        cz = np.maximum(np.log2(lin) * f32(u["scale"]) + f32(u["bias"]), 0).astype(np.int64)
    nx, ny = int(u["num_clusters"][0]), int(u["num_clusters"][1])
    cl = cz * nx * ny + cy * nx + cx
    cl = np.clip(cl, 0, len(cluster_counts) - 1)
    L = cluster_counts[cl].astype(np.int64)
    return np.where(d != 0, L, 0), d != 0


def algorithmic_work(uniforms, depth0, depth1, cluster_counts, y0, y1, width, height):
    """flops and HBM bytes per pass for rows [y0,y1) — the numerators of the roofline fractions."""
    L0, c0 = pixel_light_counts(uniforms, depth0, cluster_counts, y0, y1)
    L1, c1 = pixel_light_counts(uniforms, depth1, cluster_counts, y0, y1)
    n = (y1 - y0) * width
    n0, n1 = int(c0.sum()), int(c1.sum())
    work = {
        "shade_opaque": {"flops": float(180 * n0 + 100 * int(L0.sum())), "bytes": float(28 * n0 + 4 * (n - n0) + 16 * n)},
        "shade_transmission": {"flops": float(494 * n1 + 193 * int(L1.sum())), "bytes": float((32 + 8) * n1 + 4 * (n - n1) + 0.63 * n1)},
        "mips": {"flops": float(5 * 4 * width * height * 4 / 3), "bytes": float(width * height * (8 + 8 / 3))},  # every rank builds the whole pyramid
        "tonemap": {"flops": float(60 * n), "bytes": float(12 * n)},
        "coverage_opaque": n0 / n, "coverage_transmissive": n1 / n,
        "mean_lights_opaque": float(L0.sum() / max(n0, 1)), "mean_lights_transmissive": float(L1.sum() / max(n1, 1)),
    }
    return work


# ----------------------------------------------------------------------------- CPU oracle port (baseline + reference arm)
class CpuShadePath:
    """shader + glam-pbr per-pixel code (the oracle port) over a contiguous band of the workload's frame.

    The reference rasterises in hardware and has no CPU rasteriser, so the G-buffer of the band is an INPUT of the timed
    step: either handed in (`gbuffers`: the GPU arm passes its own planes, bit-identical to the oracle's — tests
    test_visibility_bit_exact — which makes a whole-frame baseline affordable) or produced once, untimed, by the oracle's
    software visibility pass (--impl reference: no GPU code on that path).  The timed step is fragment -> mip chain
    (prorated to the band's share of the frame) -> fragment_transmission -> tonemap."""

    def __init__(self, scene, lut, rows, opaque_full16=None, gbuffers=None):
        from oracle import pyoracle as oracle
        from transmission_renderer_b200 import abi, host
        self.oracle = oracle
        # Which code shades: the reference's own compiled shader modules (oracle/_ref/libspvref.so: its shipped SPIR-V translated to
        # C instruction by instruction, oracle/spv2c.py) when that library is here, else the C port of the same source.  The two
        # agree bit for bit (tests/test_reference_spirv.py); TR_CPU_CODE=port forces the port.
        self.code, self.code_note = "port", None
        if os.environ.get("TR_CPU_CODE", "spirv") != "port":
            try:
                from oracle import spvref
                if spvref.available():
                    spvref.lib()
                    self.spvref, self.code = spvref, "spirv"
            except Exception as e:      # noqa: BLE001 - a missing / unloadable library must not fail the bench: the port is the fallback
                self.code_note = f"reference modules not loadable ({str(e)[:120]}); the port was timed"
        # torchrun exports OMP_NUM_THREADS=1; the CPU arm is meant to use every host core it may run on
        oracle.set_num_threads(len(os.sched_getaffinity(0)))
        cam = scene["camera"]
        self.w, self.h = cam.width, cam.height
        rows = max(4, min(rows, self.h))
        self.y0 = (self.h - rows) // 2
        self.y1 = self.y0 + rows
        t = time.perf_counter()
        pc = cam.push_constants()
        if "gbuffer" in scene:                       # config 1: the synthetic G-buffer is the workload
            self.g0, self.g1, how = None, scene["gbuffer"], "synthetic G-buffer (the workload's input)"
            opaque_full16 = oracle.f16_bits(scene["opaque"])
        elif gbuffers is not None:
            (self.g0, self.g1), how = gbuffers, "G-buffer planes read back from the GPU arm (bit-identical to the oracle's rasteriser)"
        else:
            _, visible = oracle.frustum_culling(scene["instances"], scene["primitives"], cam.culling())
            self.g0, self.g1 = oracle.visibility(scene["mesh"], scene["instances"], scene["primitives"], visible, pc, self.y0, self.y1)
            how = "G-buffer by the oracle's visibility pass"
        aabbs = oracle.write_cluster_data(scene["uniforms"], cam.write_cluster_data())
        if len(scene["lights"]):
            counts, indices = oracle.assign_lights_to_clusters(scene["lights"], aabbs, cam.assign_lights())
        else:
            counts = np.zeros(len(aabbs), np.uint32)
            indices = np.zeros(len(aabbs) * abi.TR_MAX_LIGHTS_PER_CLUSTER, np.uint32)
        self.sc = dict(push_constants=pc, uniforms=scene["uniforms"], materials=scene["materials"], lights=scene["lights"],
                       cluster_light_counts=counts, cluster_light_indices=indices)
        self.lut, self.opaque_full16 = lut, opaque_full16
        self.runner = self._runner()
        self.setup_s = time.perf_counter() - t
        self.how = f"{how}, untimed ({self.setup_s:.1f} s)"
        self.cores = oracle.num_threads()

    def _runner(self):
        from transmission_renderer_b200 import host
        g0 = self.g0
        if g0 is None:   # config 1 has no opaque geometry: an empty opaque layer, the opaque frame is the procedural input
            g0 = dict(depth=np.zeros((self.h, self.w), np.float32), normal=np.zeros((self.h, self.w, 3), np.float32), uv=None,
                      material_id=np.zeros((self.h, self.w), np.uint32), scale=None, position=None)
        cls = self.spvref.ShadePathRunner if self.code == "spirv" else self.oracle.ShadePathRunner
        return cls(g0, self.g1, self.sc, self.lut, host.default_tonemap_params(), self.opaque_full16)

    @property
    def kind(self):
        """cpu_baseline.kind: "reference" = the reference's own compiled shader modules, "port" = the C restatement."""
        return "reference" if self.code == "spirv" else "port"

    def time_port(self, steps):
        """The same steps through the C port, when the primary figure is the reference's modules."""
        if self.code != "spirv":
            return None
        self.code = "port"
        try:
            self.runner = self._runner()
            self.step()
            t = float(np.median([self.step() for _ in range(steps)]))
        finally:
            self.code = "spirv"
            self.runner = self._runner()
        return self.pixels / t / 1e6

    @property
    def pixels(self):
        return (self.y1 - self.y0) * self.w

    def step(self):
        r = self.runner
        t0 = time.perf_counter()
        if self.g0 is not None:
            r.opaque(self.y0, self.y1)
        t1 = time.perf_counter()
        r.mips()
        t2 = time.perf_counter()
        r.transmission(self.y0, self.y1)
        r.tonemap(self.y0, self.y1)
        t3 = time.perf_counter()
        share = (self.y1 - self.y0) / self.h
        return (t1 - t0) + (t2 - t1) * share + (t3 - t2)

    def time_o3(self, steps):
        """The same steps through an `-O3 -march=native` build of the port (BASELINE.md 3: reported separately and labelled;
        the parity build is -O2 -ffp-contract=off).  None if that build fails on this host."""
        try:
            self.oracle.select_variant("o3")
        except Exception as e:      # noqa: BLE001 - a missing compiler flag must not fail the bench
            return None, str(e)[:200]
        code = self.code
        self.code = "port"              # the -O3 build exists for the port only
        try:
            self.runner = self._runner()
            self.step()
            t = float(np.median([self.step() for _ in range(steps)]))
        finally:
            self.oracle.select_variant("parity")
            self.code = code
            self.runner = self._runner()
        return self.pixels / t / 1e6, "gcc -O3 -march=native (contraction on): NOT the parity build"

    def describe(self):
        whole = "the whole" if (self.y0, self.y1) == (0, self.h) else f"rows [{self.y0},{self.y1}) of the"
        code = ("the reference's shipped fragment.spv / fragment_transmission.spv translated to C (oracle/spv2c.py)" if self.code == "spirv"
                else "the C port of shader + glam-pbr" + (f" [{self.code_note}]" if self.code_note else ""))
        return (f"{whole} {self.w}x{self.h} frame ({self.pixels} px): fragment -> mip chain (prorated) -> "
                f"fragment_transmission -> tonemap, shaded by {code}; {self.how}")


def cpu_sample(scene, lut, opaque_full16=None, max_pixels=500_000, gbuffers=None):
    """The bounded CPU sample: a centred band of at most `max_pixels` pixels (128 rows at 4K; one step of it is ~0.3-1 s of
    all-core CPU work, the untimed G-buffer set-up by the oracle's rasteriser ~15-20 s), or the whole frame when it is
    small enough / when the G-buffer comes from the GPU arm."""
    w, h = scene["camera"].width, scene["camera"].height
    return CpuShadePath(scene, lut, max(8, min(h, max_pixels // w)), opaque_full16, gbuffers)


def run_reference(args, wl):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    world = int(os.environ.get("WORLD_SIZE", str(args.gpus)))
    scene = make_scene(wl)
    lut = load_lut()
    # whole frame for the 512^2 / 1080p configs (BASELINE.md 3: "configs 1-3 at full size"), a bounded band above that
    cpu = cpu_sample(scene, lut, max_pixels=2_100_000 if wl["width"] * wl["height"] <= 1920 * 1080 else 500_000)
    for _ in range(args.warmup):
        cpu.step()
    times = [cpu.step() for _ in range(args.steps)]
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, cpu.runner.hdr16[cpu.y0:cpu.y1], cpu.runner.srgb8[cpu.y0:cpu.y1])
    total = float(sum(times))
    value = cpu.pixels * args.steps / total / 1e6
    line = {
        "impl": "reference", "metric": "shaded_mpixels_per_s", "value": value, "unit": "Mpx/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": total / args.steps * 1e3, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": base_config(wl, args, world),
        "cpu_baseline": {"value": value, "unit": "Mpx/s", "cores": cpu.cores, "kind": cpu.kind, "sample": cpu.describe(),
                         "value_port": cpu.time_port(max(1, args.steps // 2))},
        "e2e": {"value": value, "unit": "Mpx/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "ms_per_full_frame_extrapolated": total / args.steps * 1e3 * (wl["width"] * wl["height"]) / cpu.pixels,
        "note": "the reference's per-pixel shader code on the host cores: its shipped SPIR-V modules translated to C (kind \"reference\"; the "
                "Rust host cannot be built here), or the C port of the same source when that library is absent (kind \"port\"; the two agree "
                "bit for bit, tests/test_reference_spirv.py); ms_per_step is for the sampled rows",
    }
    print(json.dumps(line), flush=True)
    return 0


# ----------------------------------------------------------------------------- the B200 arm
def sha256_rows(arr, y0, y1):
    import hashlib
    return hashlib.sha256(np.ascontiguousarray(arr[y0:y1]).tobytes()).hexdigest()


DUMP_BYTES = 64_000_000      # --dump-outputs budget, all files together
DUMP_PIXELS = 1 << 20        # pixels kept of a frame over the budget (2 x 16 MiB of float32 RGBA)
DUMP_SEED = 0


def dump_outputs(dirname, hdr_bits, srgb):
    """Writes the frame (RGBA16F bits, sRGB8) as float32 .npy files: whole (H, W, 4) when both fit DUMP_BYTES, else the
    (DUMP_PIXELS, 4) pixels at the ascending flat indices a generator seeded with DUMP_SEED picks.

    Shaded values beyond the range of the RGBA16F target are stored there as +-inf (sun highlights of the bench scenes
    reach 5e5); they are written as +-65504, the largest finite half, as the tonemapped frame saturates them at 255."""
    os.makedirs(dirname, exist_ok=True)
    half_max = float(np.finfo(np.float16).max)
    hdr = np.clip(np.ascontiguousarray(hdr_bits).view(np.float16).astype(np.float32), -half_max, half_max)
    out = np.asarray(srgb, np.float32)
    h, w = hdr.shape[:2]
    if 2 * hdr.nbytes > DUMP_BYTES:
        keep = np.sort(np.random.default_rng(DUMP_SEED).choice(h * w, DUMP_PIXELS, replace=False))
        hdr, out = hdr.reshape(-1, 4)[keep], out.reshape(-1, 4)[keep]
    np.save(os.path.join(dirname, "hdr_rgba.npy"), hdr)
    np.save(os.path.join(dirname, "srgb8_rgba.npy"), out)


def run_b200(args, wl):
    import torch
    import torch.distributed as dist
    from transmission_renderer_b200 import Renderer, abi, host, parallel, scenes

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("bench.py --gpus N > 1 must be launched with torch.distributed.run (one rank per GPU)")
        args.gpus = world
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the product has no CPU path (use --impl reference for the CPU port)")
    torch.cuda.set_device(local_rank)
    cpu_group = None
    if world > 1:
        dist.init_process_group(backend="nccl", device_id=torch.device("cuda", local_rank))
        cpu_group = dist.new_group(backend="gloo")

    def barrier():
        if world > 1:
            dist.barrier(group=cpu_group)

    W, H = wl["width"], wl["height"]
    synthetic = wl["kind"] == "config1"          # configs[0]: the G-buffer and the opaque frame are the inputs
    if synthetic and (world > 1 or args.views > 1 or args.ray_tracing):
        raise SystemExit("--workload config1 is the single-GPU, single-view synthetic-G-buffer case")
    scene = make_scene(wl)
    if "instances" in scene:   # the exact #[repr(C)] layout (48-byte Instance), whatever dtype the scene builder concatenated
        scene["instances"] = np.ascontiguousarray(scene["instances"]).astype(abi.instance)
        scene["lights"] = np.ascontiguousarray(scene["lights"]).astype(abi.light)
    lut = load_lut()
    cam = scene["camera"]
    stream = torch.cuda.Stream()
    r = Renderer(W, H, device=local_rank)
    r.set_stream(stream.cuda_stream)
    r.set_uniforms(scene["uniforms"])
    r.set_materials(scene["materials"])
    r.set_lights(scene["lights"])
    r.set_ggx_lut(lut)
    tm = host.default_tonemap_params()
    pc = cam.push_constants()
    if synthetic:
        opaque_bits = np.asarray(scene["opaque"], np.float32).astype(np.float16).view(np.uint16)   # RGBA16F, round to nearest even
        r.build_clusters(cam.write_cluster_data())
        r.assign_lights(cam.assign_lights())
        r.set_gbuffer(abi.TR_LAYER_TRANSMISSIVE, scene["gbuffer"])
        r.set_opaque_frame(opaque_bits)
    else:
        r.set_instances(scene["instances"])
        r.set_primitives(scene["primitives"])
        m = scene["mesh"]
        r.set_mesh(m["positions"], m["normals"], m["uvs"], m["indices"])
        r.build_clusters(cam.write_cluster_data())
    as_handle, as_build_ms = 0, None
    if args.ray_tracing:                          # the reference's `--ray-tracing` option (src/main.rs:84, 577-658)
        t0 = time.perf_counter()
        as_handle = r.build_acceleration_structures()
        as_build_ms = (time.perf_counter() - t0) * 1e3
    groups = max(1, min(args.view_groups, world))
    if world % groups or args.views % groups:
        raise SystemExit("--view-groups must divide both the GPU count and --views")
    bands = world // groups                      # ranks per view group = bands per frame
    group_id, band_rank = rank // bands, rank % bands
    band_group = cpu_group
    if groups > 1 and bands > 1:                 # one gloo group per view group for the unique-id / IPC-handle exchange
        for g in range(groups):
            sub = dist.new_group(ranks=list(range(g * bands, (g + 1) * bands)), backend="gloo")
            if g == group_id:
                band_group = sub
    parallel.init_bands(r, band_rank, bands, group=band_group, exchange=args.exchange)
    y0, y1 = host.band_rows(H, band_rank, bands)
    if args.emulate_band and world == 1:
        eb_r, eb_n = (int(x) for x in args.emulate_band.split("/"))
        y0, y1 = host.band_rows(H, eb_r, eb_n)
        r.set_band(y0, y1)
    fp = cam.frame_params(tm, acceleration_structure_address=as_handle)
    # views of this rank's group: orbit in yaw around the scene centre (configs[4]); view 0 is the scene's own camera
    my_fps = [fp]
    if args.views > 1:
        my_fps = []
        for v in range(group_id, args.views, groups):
            vc = scenes.Camera(W, H, tuple(cam.position), 360.0 * v / args.views, -10.0)
            my_fps.append(vc.frame_params(tm, acceleration_structure_address=as_handle))
    frames_per_step = len(my_fps)

    def one_step():
        if synthetic:                            # configs[0]: mip chain of the given opaque frame -> fragment_transmission -> tonemap
            r.begin_frame()
            r.generate_mips()
            r.shade_transmission(pc)
            r.tonemap(tm)
        else:
            for f in my_fps:
                r.frame(f)

    def sync():
        stream.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()

    # N > 1: equal-row bands leave the ranks unequal work (coverage, triangle density and light counts vary down the frame);
    # a few untimed frames with the per-pass timers on move the boundaries until every band costs about the same. The frame
    # is bitwise the same for any boundaries (frame_sha256 below).
    band_bounds = [host.band_rows(H, b, bands)[0] for b in range(bands)] + [H]
    if bands > 1 and not args.equal_bands and not args.emulate_band:
        with torch.cuda.stream(stream):
            for _ in range(3):
                one_step()
            sync()
            band_bounds = parallel.balance_bands(r, lambda: [one_step() for _ in range(3)], band_rank, bands, group=band_group)
        y0, y1 = band_bounds[band_rank], band_bounds[band_rank + 1]

    # the 512^2 case fits L2: a 256 MB buffer is overwritten between timed steps, each step under its own event pair
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda") if W * H < 1920 * 1080 else None

    def timed_steps(n):
        """device time of n steps (ms), max over ranks; events on the launch stream"""
        if flush is None:
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record(stream)
            for _ in range(n):
                one_step()
            ev1.record(stream)
            sync()
            return ev0.elapsed_time(ev1)
        pairs = []
        for _ in range(n):
            flush.fill_(1)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            one_step()
            e1.record(stream)
            pairs.append((e0, e1))
        sync()
        return float(sum(a.elapsed_time(b) for a, b in pairs))

    # ------------------------------------------------------------------ resident: inputs already in HBM
    with torch.cuda.stream(stream):
        for _ in range(max(args.warmup, 3)):
            one_step()
        sync()
        r.enable_timing(True)
        launches0 = Renderer.launch_count()
        barrier()
        sync()
        t_wall0 = time.time()
        ms_local = timed_steps(args.steps)
        t_wall1 = time.time()
        barrier()
        ms_total = max_over_ranks(ms_local)
        launches = Renderer.launch_count() - launches0
        totals, n_timed = r.pass_totals()
        rstats = r.raster_stats()
        r.enable_timing(False)
        # ---- sustained: the same steps back to back for >= --min-seconds, its own clock window
        sustained = None
        if args.min_seconds > 0:
            chunks = max(1, int(np.ceil(args.min_seconds * 1e3 / max(ms_total, 1e-3))))
            barrier()
            sync()
            s_wall0 = time.time()
            s_ms = sum(timed_steps(args.steps) for _ in range(chunks))
            s_wall1 = time.time()
            barrier()
            s_ms = max_over_ranks(s_ms)
            sustained = {"value": W * H * args.views * args.steps * chunks / (s_ms * 1e-3) / 1e6, "unit": "Mpx/s",
                         "steps": args.steps * chunks, "seconds": s_ms * 1e-3, "ms_per_step": s_ms / (args.steps * chunks)}
    ms_per_step = ms_total / args.steps
    value = W * H * args.views / (ms_per_step * 1e-3) / 1e6
    passes = {k[:-3]: v / max(n_timed, 1) for k, v in totals.items()}
    if sampler:
        clocks = sampler.summary(t_wall0, t_wall1)
        if clocks["samples"] == 0:
            clocks = sampler.summary()
        if sustained is not None:
            sc = sampler.summary(s_wall0, s_wall1)
            sustained["clocks"] = {k: sc.get(k) for k in ("sm_mhz", "sm_max_mhz", "reasons", "samples", "power_w_max")}

    # ------------------------------------------------------------------ end to end: host buffers in, sRGB8 band out
    out_pinned = [torch.empty(H * W * 4, dtype=torch.uint8).pin_memory() for _ in range(2)]
    out_host = [o.numpy().reshape(H, W, 4) for o in out_pinned]
    d2h = (y1 - y0) * W * 4
    e2e_skip = set(filter(None, os.environ.get("TR_E2E_SKIP", "").split(",")))   # diagnosis only: inst, lights, readback
    if synthetic:
        # the reference-facing call of this case takes the G-buffer planes and the opaque frame as HOST buffers
        def pin(a):
            t = torch.empty(a.nbytes, dtype=torch.uint8).pin_memory()
            v = t.numpy().view(a.dtype).reshape(a.shape)
            v[...] = a
            return t, v
        keep = {k: pin(np.ascontiguousarray(v)) for k, v in scene["gbuffer"].items() if v is not None}
        g_host = {k: (keep[k][1] if k in keep else None) for k in scene["gbuffer"]}
        o_keep = pin(opaque_bits)
        h2d = sum(v[1].nbytes for v in keep.values()) + o_keep[1].nbytes

        def e2e_step(j):
            r.set_gbuffer(abi.TR_LAYER_TRANSMISSIVE, g_host)
            r.set_opaque_frame(o_keep[1])
            one_step()
            r.read_srgb8_async(out_host[j & 1])
    else:
        inst_pinned = torch.empty(scene["instances"].nbytes, dtype=torch.uint8).pin_memory()
        inst_host = inst_pinned.numpy().view(abi.instance)
        inst_host[:] = scene["instances"]
        lights_pinned = torch.empty(max(scene["lights"].nbytes, 48), dtype=torch.uint8).pin_memory()
        lights_host = lights_pinned.numpy()[:scene["lights"].nbytes].view(abi.light)
        lights_host[:] = scene["lights"]
        h2d = inst_host.nbytes + lights_host.nbytes + fp.nbytes

        def e2e_step(j):
            # frame i: inputs up, frame, band read-back enqueued behind it on the copy stream; then hand frame i-1's band
            # (other pinned buffer) to the consumer — like the reference presenting frame n-1 while recording frame n
            for k, f in enumerate(my_fps):
                i = j * frames_per_step + k
                if "inst" not in e2e_skip:
                    r.set_instances(inst_host)
                if "lights" not in e2e_skip:
                    r.set_lights(lights_host)
                if args.ray_tracing:     # an instance write is followed by the top-level update, src/main.rs:1263-1345
                    f["push_constants"]["acceleration_structure_address"] = r.update_top_level_acceleration_structure()
                r.frame(f)
                if "readback" not in e2e_skip:
                    r.read_srgb8_async(out_host[i & 1])

    with torch.cuda.stream(stream):
        for i in range(max(args.warmup, 3)):
            e2e_step(i)
        r.sync()
        barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record(stream)
        t_host = time.perf_counter()
        for i in range(args.steps):
            e2e_step(i)
        host_submit_ms = (time.perf_counter() - t_host) * 1e3 / args.steps   # host time to ENQUEUE a step (no waiting in it)
        r.wait_readback()            # the last band is on the host before the clock stops
        ev1.record(stream)
        sync()
        barrier()
        e2e_ms = max_over_ranks(ev0.elapsed_time(ev1)) / args.steps
    e2e_value = W * H * args.views / (e2e_ms * 1e-3) / 1e6
    if sampler:
        sampler.stop()

    # ------------------------------------------------------------------ band hashes: N-GPU output == 1-GPU output, from the lines
    band_hashes, frame_sha = None, None
    frame = None   # rank 0: (RGBA16F bits, sRGB8) of the whole frame of the last step, for --dump-outputs
    if args.views == 1 and not args.emulate_band:
        hdr_bits, srgb = r.read_hdr(), r.read_srgb8()
        mine = {"rows": [int(y0), int(y1)], "hdr_rgba16f": sha256_rows(hdr_bits, y0, y1), "srgb8": sha256_rows(srgb, y0, y1)}
        if world > 1:
            every = [None] * world
            dist.all_gather_object(every, mine, group=cpu_group)
            band_hashes = {str(bands): every[:bands]}
            if groups == 1:   # the whole frame, stitched from the ranks' bands on rank 0 (outside every timed region)
                parts = [None] * world
                dist.all_gather_object(parts, (hdr_bits[y0:y1].copy(), srgb[y0:y1].copy()), group=cpu_group)
                if rank == 0:
                    import hashlib
                    frame_sha = {"hdr_rgba16f": hashlib.sha256(b"".join(p[0].tobytes() for p in parts)).hexdigest(),
                                 "srgb8": hashlib.sha256(b"".join(p[1].tobytes() for p in parts)).hexdigest()}
                    frame = (np.concatenate([p[0] for p in parts]), np.concatenate([p[1] for p in parts]))
        else:
            frame = (hdr_bits, srgb)
            frame_sha = {"hdr_rgba16f": sha256_rows(hdr_bits, 0, H), "srgb8": sha256_rows(srgb, 0, H)}
            band_hashes = {}
            for n in (1, 2, 4, 8):
                rows = [host.band_rows(H, b, n) for b in range(n)]
                band_hashes[str(n)] = [{"rows": [int(a), int(b)], "hdr_rgba16f": sha256_rows(hdr_bits, a, b), "srgb8": sha256_rows(srgb, a, b)}
                                       for a, b in rows]
    if args.dump_outputs and rank == 0:
        if frame is None:   # several views a step, view groups or an emulated band: rank 0's rows of its last frame
            frame = (r.read_hdr()[y0:y1], r.read_srgb8()[y0:y1])
        dump_outputs(args.dump_outputs, *frame)

    # ------------------------------------------------------------------ roofline of the dominant pass (rank 0's band)
    line = None
    if rank == 0:
        g1 = r.read_gbuffer(1)
        g0 = r.read_gbuffer(0) if not synthetic else dict(depth=np.zeros((H, W), np.float32))
        n_clusters = int(scene["uniforms"]["num_clusters"][0, 0]) * int(scene["uniforms"]["num_clusters"][0, 1]) * 16
        cc, _ = r.read_cluster_lights(n_clusters)
        work = algorithmic_work(scene["uniforms"], g0["depth"].reshape(H, W), g1["depth"].reshape(H, W), cc, y0, y1, W, H)
        if not synthetic:   # K1-K3 (SURVEY.md 8d bytes; visibility: DESIGN.md 4)
            vis_ids = r.read_visible_instances()
            prim_tris = scene["primitives"]["index_count"][scene["instances"]["primitive_id"][vis_ids]] // 3
            n_inst, n_prim = len(scene["instances"]), len(scene["primitives"])
            n_draws = int(sum(len(r.read_draws(b)) for b in range(4)))
            work["cull"] = {"flops": 60.0 * n_inst, "bytes": float(48 * n_inst + 32 * n_prim + 4 * len(vis_ids) + 4 * n_prim + 20 * n_draws)}
            work["assign_lights"] = {"flops": 40.0 * n_clusters * len(scene["lights"]),
                                     "bytes": float(48 * len(scene["lights"]) + 32 * n_clusters + 4 * n_clusters + 4 * int(cc.sum()))}
            n_band = (y1 - y0) * W
            work["visibility"] = {"flops": 0.0, "bytes": float((60 + 2 * 2 * 8) * n_band + (12 + 3 * 32) * int(prim_tris.sum()))}
        hbm_peak, hbm_src = measured_peaks()
        fp32_peak = r.measure_fp32_peak()
        names = ("shade_opaque", "mips", "shade_transmission", "tonemap") if synthetic else \
            ("cull", "assign_lights", "visibility", "shade_opaque", "mips", "shade_transmission", "tonemap")
        shade = {k: passes[k] for k in names}
        kernels = {}
        for k, ms in shade.items():
            wk = work[k]
            gbs = wk["bytes"] / (ms * 1e-3) / 1e9 if ms > 0 else 0.0
            tfl = wk["flops"] / (ms * 1e-3) / 1e12 if ms > 0 else 0.0
            kernels[k] = {"ms": ms, "GB/s": gbs, "hbm_frac": gbs / hbm_peak, "TFLOP/s": tfl, "fp32_frac": tfl / fp32_peak}
        # the dominant KERNEL: cull / assign_lights / visibility are passes of several small kernels each (visibility: six),
        # listed under `kernels` with the pass's bytes; the roofline object is for the longest single kernel
        dom = max(("shade_opaque", "mips", "shade_transmission", "tonemap"), key=lambda k: shade[k])
        kd = kernels[dom]
        traffic, traffic_src = ncu_traffic(dom, args.workload, world)
        if kd["fp32_frac"] >= kd["hbm_frac"]:
            roofline = {"kernel": dom, "bound": "fp32", "achieved": kd["TFLOP/s"], "peak": fp32_peak, "unit": "TFLOP/s",
                        "frac": kd["fp32_frac"], "traffic": traffic, "traffic_source": traffic_src,
                        "peak_source": "FFMA-chain microbenchmark in this run (MEASURED_PEAKS.json has no FP32 figure; nominal 74.4)"}
        else:
            roofline = {"kernel": dom, "bound": "hbm", "achieved": kd["GB/s"], "peak": hbm_peak, "unit": "GB/s",
                        "frac": kd["hbm_frac"], "traffic": traffic, "traffic_source": traffic_src, "peak_source": hbm_src}
        shade_path_ms = passes["shade_opaque"] + passes["allgather"] + passes["mips"] + passes["shade_transmission"]
        line = {
            "metric": "shaded_mpixels_per_s", "value": value, "unit": "Mpx/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": base_config(wl, args, world),
            "workload_stats": {"coverage_opaque": work["coverage_opaque"], "coverage_transmissive": work["coverage_transmissive"],
                               "mean_lights_opaque": work["mean_lights_opaque"], "mean_lights_transmissive": work["mean_lights_transmissive"]},
            "clocks": {k: clocks[k] for k in ("sm_mhz", "sm_max_mhz", "reasons")} | {"samples": clocks["samples"]},
            "e2e": {"value": e2e_value, "unit": "Mpx/s", "ms_per_step": e2e_ms, "h2d_bytes_per_step": int(h2d) * frames_per_step,
                    "d2h_bytes_per_step": int(d2h) * frames_per_step, "host_submit_ms_per_step": host_submit_ms},
            "gpu_launches": int(launches),
            "sustained": sustained,
            "passes_ms": passes,
            "kernels": kernels,
            "roofline": roofline,
            "shade_path": {"ms": shade_path_ms, "Mpx/s": W * H / (shade_path_ms * 1e-3) / 1e6},
            "fp32_peak_tflops_measured": fp32_peak,
            "raster_stats_per_frame": {k: v / (args.steps + max(args.warmup, 3)) for k, v in rstats.items()},
            "band_rows": [int(v) for v in band_bounds],
            "frame_sha256": frame_sha,
            "band_hashes": band_hashes,
        }
        # ---- CPU baseline: the oracle port on the box's host cores, bounded sample, N=1 only; doubles as a live parity check
        if as_build_ms is not None:
            line["acceleration_structure_build_ms"] = as_build_ms
            line["roofline"]["note"] = "shading passes include the shadow-ray pass; its traversal work is not in the algorithmic flop count"
        if world == 1 and args.views == 1 and not args.no_cpu_baseline and not args.ray_tracing and not args.emulate_band:
            opaque16 = r.read_pyramid_level(0)
            gpu_hdr = r.read_hdr()
            # the whole frame up to 4K (the G-buffer comes from the GPU arm: no CPU rasterisation needed), a band at 8K
            whole = W * H <= 3840 * 2160
            cpu = cpu_sample(scene, lut, opaque16, max_pixels=W * H if whole else 500_000, gbuffers=(g0, g1) if (whole and not synthetic) else None)
            cpu.step()
            n_cpu = int(np.clip(round(12.0 / max(cpu.step(), 1e-3)), 2, 15))   # ~10-20 s of all-core CPU work
            times = [cpu.step() for _ in range(n_cpu)]
            best = float(np.median(times))
            from oracle import pyoracle as oracle
            a = oracle.f16_to_f32(gpu_hdr[cpu.y0:cpu.y1])[..., :3].astype(np.float64)
            b = oracle.f16_to_f32(cpu.runner.hdr16[cpu.y0:cpu.y1])[..., :3].astype(np.float64)
            ok = np.isfinite(a) & np.isfinite(b)
            rel = float(np.linalg.norm(a[ok] - b[ok]) / max(np.linalg.norm(b[ok]), 1e-30))
            line["cpu_baseline"] = {"value": cpu.pixels / best / 1e6, "unit": "Mpx/s", "cores": cpu.cores, "kind": cpu.kind,
                                    "sample": cpu.describe(), "steps": n_cpu, "ms_per_step": best * 1e3,
                                    "parity_rel_l2_vs_gpu": rel, "value_port": cpu.time_port(max(2, n_cpu // 3))}
            o3, o3_note = cpu.time_o3(max(2, n_cpu // 3))
            line["cpu_baseline"]["value_o3_march_native"] = o3
            line["cpu_baseline"]["o3_note"] = o3_note
    r.close()
    if world > 1:
        dist.destroy_process_group()
    if line is not None:
        print(json.dumps(line), flush=True)
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="4k", choices=sorted(WORKLOADS))
    ap.add_argument("--exchange", default="peer", choices=["nccl", "peer"],
                    help="N>1: opaque bands by fused peer stores over NVLink (default) or by an NCCL all-gather")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--ray-tracing", action="store_true",
                    help="ray-queried shadows on (the reference's --ray-tracing option); off for the headline metric")
    ap.add_argument("--min-seconds", type=float, default=0.0,
                    help="also run the timed steps back to back for at least this long and report `sustained` (0 = off, the default)")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="after the timed steps, write the frame of the last step to DIR/*.npy (float32; sampled above 64 MB)")
    ap.add_argument("--views", type=int, default=None,
                    help="camera views per step (BASELINE configs[4]: 64 orbit views, the default of --workload config5); a step renders all of them")
    ap.add_argument("--view-groups", type=int, default=1,
                    help="N ranks = view-groups x bands: each group of N/view-groups ranks renders its share of the views band-parallel")
    ap.add_argument("--equal-bands", action="store_true",
                    help="N>1: keep the equal-row bands of tr_comm_init instead of balancing the band boundaries by measured cost")
    ap.add_argument("--emulate-band", default=None, metavar="R/N",
                    help="profiling aid (1 GPU): render only band R of N without any exchange, e.g. 3/8")
    args = ap.parse_args()
    wl = WORKLOADS[args.workload]
    if args.views is None:
        args.views = wl.get("views", 1)
    if args.impl == "reference":
        return run_reference(args, wl)
    return run_b200(args, wl)


if __name__ == "__main__":
    sys.exit(main())
