"""bench.py contract, the parts that run without a GPU: the reference arm prints one JSON line with the keys the driver reads,
and the product arm refuses to run without a CUDA device instead of falling back to anything."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args, **env):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=600,
                          env=dict(os.environ, CUDA_VISIBLE_DEVICES="", **env))


@pytest.mark.parametrize("code", ["spirv", "port"])
def test_reference_arm_line(code):
    """code = spirv: the reference's own compiled shader modules shade (oracle/_ref/libspvref.so; kind "reference", or "port"
    with a note where that library is absent); code = port: the C restatement is forced (TR_CPU_CODE=port)."""
    p = _run("--impl", "reference", "--steps", "1", "--warmup", "0", TR_CPU_CODE=code)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "shaded_mpixels_per_s" and d["unit"] == "Mpx/s" and d["higher_is_better"] is True
    assert d["n_gpus"] == 1 and d["steps"] == 1 and d["value"] > 0 and d["ms_per_step"] > 0
    assert d["config"]["workload"].startswith("configs[3]") and d["config"]["width"] == 3840 and d["config"]["lights"] == 64
    cb = d["cpu_baseline"]
    from oracle import build_ref
    kind = "reference" if code == "spirv" and build_ref.build() is not None else "port"
    assert cb["kind"] == kind and cb["cores"] >= 1 and cb["value"] == d["value"] and "rows" in cb["sample"]
    assert (cb["value_port"] is not None and cb["value_port"] > 0) == (kind == "reference")
    assert ("fragment.spv" in cb["sample"]) == (kind == "reference")
    assert d["e2e"] == {"value": d["value"], "unit": "Mpx/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_dump_outputs_of_the_reference_arm(tmp_path):
    """--dump-outputs: the last timed step's frame as float32 .npy files, the same bytes from run to run."""
    dumps = []
    for run in ("a", "b"):
        p = _run("--impl", "reference", "--workload", "config1", "--steps", "2", "--warmup", "0", "--dump-outputs", str(tmp_path / run))
        assert p.returncode == 0, p.stderr[-2000:]
        dumps.append({n: np.load(tmp_path / run / f"{n}.npy") for n in ("hdr_rgba", "srgb8_rgba")})
    for n, a in dumps[0].items():
        assert a.dtype == np.float32 and a.shape == (512, 512, 4), n
        assert np.isfinite(a).all(), n
        assert a.tobytes() == dumps[1][n].tobytes(), n
    srgb, hdr = dumps[0]["srgb8_rgba"], dumps[0]["hdr_rgba"]
    assert srgb.max() <= 255 and np.array_equal(srgb, np.round(srgb)) and srgb[..., :3].mean() > 0
    # config 1's sun highlight overflows the RGBA16F target: written as the largest finite half, saturated in sRGB8
    over = hdr[..., :3] == 65504
    assert over.any() and (srgb[..., :3][over] == 255).all()


def test_dump_outputs_samples_a_large_frame(tmp_path):
    """A frame over the 64 MB budget: the same seeded pixels every time, the files within the budget."""
    import bench
    rng = np.random.default_rng(1)
    h, w = 1080, 1920
    values = rng.uniform(0, 8, (h, w, 4))
    values[rng.random((h, w, 4)) < 0.1] = 1e6            # overflows the half range: stored as inf
    with np.errstate(over="ignore"):
        hdr = values.astype(np.float16).view(np.uint16)
    srgb = rng.integers(0, 256, (h, w, 4), dtype=np.uint8)
    bench.dump_outputs(str(tmp_path), hdr, srgb)
    a, b = np.load(tmp_path / "hdr_rgba.npy"), np.load(tmp_path / "srgb8_rgba.npy")
    assert a.shape == b.shape == (bench.DUMP_PIXELS, 4) and a.dtype == b.dtype == np.float32
    assert np.isfinite(a).all() and np.isfinite(b).all()
    assert sum(os.path.getsize(tmp_path / f) for f in os.listdir(tmp_path)) <= bench.DUMP_BYTES
    keep = np.sort(np.random.default_rng(bench.DUMP_SEED).choice(h * w, bench.DUMP_PIXELS, replace=False))
    expect = hdr.view(np.float16).reshape(-1, 4)[keep].astype(np.float32)
    assert np.isinf(expect).any()
    assert np.array_equal(a, np.where(np.isinf(expect), np.float32(65504), expect))
    assert np.array_equal(b, srgb.reshape(-1, 4)[keep].astype(np.float32))


def test_product_arm_needs_cuda():
    p = _run("--steps", "1", "--warmup", "0")
    assert p.returncode != 0
    assert "no CUDA device" in (p.stderr + p.stdout)
