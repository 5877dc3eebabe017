"""The rule by which tr_set_texture_async builds a mip chain on the device (csrc/k_textures.cu), restated in numpy and held
against the Python ingest's CPU chain, scenes.make_mips, which the blocking tr_set_texture is fed: the two must give the
same bytes, so that an image bound from level 0 samples bit for bit as the ingested one.

The device rule: float64 decode tables built with libm pow (math.pow here), the 2x2 box summed ((a + b) + c) + d and
multiplied by 0.25, UNORM bytes floor(clip(x) * 255 + 0.5), sRGB colour bytes = the number of 255 encode thresholds <= x.

numpy's vectorised pow is not libm's on every host (with AVX-512 it may differ by one ulp), so make_mips's decoded values and
encode decisions can differ from libm's by one ulp.  The bytes are compared in-process; the bit-level identities before
quantisation are checked in a subprocess with numpy's AVX-512 dispatch switched off, where np.power is libm's."""
import math
import os
import struct
import subprocess
import sys

import numpy as np
import pytest

from transmission_renderer_b200 import host, scenes

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ------------------------------------------------------------------------------------------------ restatement of the rule
def _srgb8_to_linear(v):
    x = v / 255.0
    return x / 12.92 if x <= 0.04045 else math.pow((x + 0.055) / 1.055, 2.4)


def _encode_byte(x):   # scenes.srgb_encode of one value, libm pow
    x = min(max(x, 0.0), 1.0)
    s = x * 12.92 if x <= 0.0031308 else 1.055 * math.pow(x, 1 / 2.4) - 0.055
    return math.floor(s * 255.0 + 0.5)


def _bits(x):
    return struct.unpack("<q", struct.pack("<d", x))[0]


def _double(b):
    return struct.unpack("<d", struct.pack("<q", b))[0]


def _thresholds():
    """encode[k - 1]: the least double in [0, 1] whose sRGB byte is >= k (bisection on the bit patterns)."""
    out = []
    for k in range(1, 256):
        lo, hi = 0, _bits(1.0)
        while hi - lo > 1:
            mid = (lo + hi) // 2
            if _encode_byte(_double(mid)) >= k:
                hi = mid
            else:
                lo = mid
        out.append(_double(hi))
    return np.array(out)


DEC_SRGB = np.array([_srgb8_to_linear(v) for v in range(256)])
DEC_UNORM = np.arange(256) / 255.0
ENCODE = _thresholds()


def box_mean(dec):
    """The device's 2x2 box over the even-cropped (h, w, 4) float64 image."""
    h, w = dec.shape[0] // 2, dec.shape[1] // 2
    s = dec[: 2 * h, : 2 * w]
    a, b, c, d = s[0::2, 0::2], s[0::2, 1::2], s[1::2, 0::2], s[1::2, 1::2]
    return (((a + b) + c) + d) * 0.25


def device_chain(rgba8, srgb, n_levels=0):
    """The byte levels tr_set_texture_async builds from level 0."""
    n = n_levels or host.mip_levels_for_size(rgba8.shape[1], rgba8.shape[0])
    levels = [np.ascontiguousarray(rgba8, np.uint8)]
    for _ in range(1, n):
        src = levels[-1]
        dec = DEC_UNORM[src]
        if srgb:
            dec[..., :3] = DEC_SRGB[src[..., :3]]
        m = box_mean(dec)
        out = np.floor(np.clip(m, 0.0, 1.0) * 255.0 + 0.5).astype(np.uint8)
        if srgb:
            out[..., :3] = np.searchsorted(ENCODE, m[..., :3], side="right").astype(np.uint8)
        levels.append(out)
    return levels


# ------------------------------------------------------------------------------------------------ images
SIZES = [(1, 1), (2, 1), (3, 3), (7, 5), (64, 64), (256, 128), (1000, 600), (2048, 2048)]   # width x height


def image(kind, w, h, seed=7):
    if kind == "random":
        return np.random.default_rng(seed + w * 131 + h).integers(0, 256, (h, w, 4), dtype=np.uint8)
    if kind == "gradient":
        y, x = np.mgrid[0:h, 0:w]
        fx, fy = x / max(w - 1, 1), y / max(h - 1, 1)
        img = np.stack([fx, fy, (fx + fy) / 2, 1.0 - fx * fy], -1)
        return np.floor(img * 255.0 + 0.5).astype(np.uint8)
    return np.broadcast_to(np.array([200, 17, 128, 77], np.uint8), (h, w, 4)).copy()


@pytest.mark.parametrize("kind", ["random", "gradient", "constant"])
@pytest.mark.parametrize("srgb", [True, False], ids=["srgb", "unorm"])
@pytest.mark.parametrize("size", SIZES, ids=[f"{w}x{h}" for w, h in SIZES])
def test_device_rule_equals_make_mips(size, srgb, kind):
    w, h = size
    img = image(kind, w, h)
    want = scenes.make_mips(img, srgb)
    got = device_chain(img, srgb)
    assert len(got) == len(want) == host.mip_levels_for_size(w, h)
    for k, (g, r) in enumerate(zip(got, want)):
        assert g.shape == r.shape, k
        assert g.tobytes() == r.tobytes(), f"level {k}: {(g != r).any(-1).sum()} texels differ"


def test_summation_order_is_numpys():
    """make_mips's mean(axis=(1, 3)) adds the 2x2 block as ((a + b) + c) + d: the restated sum is bit-equal on the same
    decoded inputs, and the other orders are not."""
    rng = np.random.default_rng(3)
    for h, w in ((64, 64), (37, 90), (600, 1000)):
        lin = scenes.srgb_decode(rng.integers(0, 256, (h, w, 4)))
        hh, ww = h // 2, w // 2
        ref = lin[: 2 * hh, : 2 * ww].reshape(hh, 2, ww, 2, 4).mean(axis=(1, 3))
        assert box_mean(lin).tobytes() == ref.tobytes()
        s = lin[: 2 * hh, : 2 * ww]
        a, b, c, d = s[0::2, 0::2], s[0::2, 1::2], s[1::2, 0::2], s[1::2, 1::2]
        assert ((((a + c) + b) + d) / 4.0 != ref).any()
        assert (((a + b) + (c + d)) / 4.0 != ref).any()


def test_decode_table_is_srgb_decode():
    """libm's decode table against scenes.srgb_decode: at most one ulp apart (numpy's pow may be a SIMD one)."""
    ref = scenes.srgb_decode(np.arange(256))
    assert np.abs(DEC_SRGB.view(np.int64) - ref.view(np.int64)).max() <= 1
    assert DEC_UNORM.tobytes() == (np.arange(256).astype(np.float64) / 255.0).tobytes()


def test_thresholds_reproduce_srgb_encode():
    """At every threshold and at its two neighbouring doubles the count of thresholds <= x is the encode formula's byte
    (libm pow); scenes.srgb_encode gives the same byte wherever its pow agrees with libm's."""
    assert (np.diff(ENCODE) > 0).all() and ENCODE[0] > 0.0 and ENCODE[-1] <= 1.0
    pts = np.concatenate([ENCODE, np.nextafter(ENCODE, 0.0), np.nextafter(ENCODE, 2.0)])
    count = np.searchsorted(ENCODE, pts, side="right")
    assert all(_encode_byte(float(x)) == k for x, k in zip(pts, count))
    assert (count[:255] == np.arange(1, 256)).all() and (count[255:510] == np.arange(0, 255)).all()
    numpy_bytes = scenes.srgb_encode(pts)
    pow_differs = np.array([np.power(x, 1 / 2.4) != math.pow(x, 1 / 2.4) for x in pts])
    assert ((numpy_bytes == count) | pow_differs).all()
    x = np.random.default_rng(5).random(1_000_000)
    assert (scenes.srgb_encode(x) == np.searchsorted(ENCODE, x, side="right")).all()


_LIBM_NUMPY = r"""
import math, sys
import numpy as np
sys.path.insert(0, sys.argv[1])
sys.path.insert(0, sys.argv[2])
from test_texture_chain_rule import DEC_SRGB, ENCODE, box_mean, device_chain, image
from transmission_renderer_b200 import scenes
assert all(np.power(x, 2.4) == math.pow(x, 2.4) for x in np.linspace(0.05, 1.0, 1001)), "np.power is not libm's here"
assert scenes.srgb_decode(np.arange(256)).tobytes() == DEC_SRGB.tobytes()
pts = np.concatenate([ENCODE, np.nextafter(ENCODE, 0.0), np.nextafter(ENCODE, 2.0)])
assert (scenes.srgb_encode(pts) == np.searchsorted(ENCODE, pts, side="right")).all()
for kind in ("random", "gradient"):
    img = image(kind, 256, 128)
    lin = img.astype(np.float64) / 255.0
    lin[..., :3] = scenes.srgb_decode(img[..., :3])
    dec = DEC_SRGB[img]
    dec[..., 3] = img[..., 3] / 255.0
    assert box_mean(dec).tobytes() == lin.reshape(64, 2, 128, 2, 4).mean(axis=(1, 3)).tobytes()
    for g, r in zip(device_chain(img, True), scenes.make_mips(img, True)):
        assert g.tobytes() == r.tobytes()
print("ok")
"""


def test_bit_identities_with_libm_pow_in_numpy():
    """With numpy's AVX-512 dispatch off, np.power is libm's: then the decode table is srgb_decode bit for bit, the
    thresholds reproduce srgb_encode exactly, and the device's float64 means equal make_mips's before quantisation."""
    from numpy._core._multiarray_umath import __cpu_features__ as feats
    env = dict(os.environ)
    off = [f for f, on in feats.items() if on and f.startswith("AVX512")]
    if off:
        env["NPY_DISABLE_CPU_FEATURES"] = " ".join(off)
    r = subprocess.run([sys.executable, "-c", _LIBM_NUMPY, ROOT, os.path.join(ROOT, "tests")], env=env,
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and r.stdout.strip().endswith("ok"), r.stdout + r.stderr
