"""Builds transmission_renderer_b200/libtr.so (sm_100a) in-tree with nvcc.

    python -m transmission_renderer_b200.csrc.build [--force] [--verbose]
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.dirname(HERE)
OUT = os.path.join(PKG, "libtr.so")
SOURCES = ["tr_api.cu", "tr_comm.cu", "tr_group.cu", "k_shade.cu", "k_shade_shadow.cu", "k_accel.cu", "k_accel_device.cu", "k_accel_build.cu", "k_mesh_update.cu", "k_instances.cu", "k_textures.cu", "k_mips.cu", "k_tonemap.cu", "k_eval.cu",
           "k_cull.cu", "k_clusters.cu", "k_visibility.cu", "k_peak.cu"]
HEADERS = ["tr_internal.h", "tr_device_math.cuh", "tr_device_pbr.cuh", "tr_device_accel.cuh", "tr_device_build.cuh",
           os.path.join("..", "..", "include", "tr_abi.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-Xcompiler",
              "-fPIC,-fvisibility=hidden,-ffp-contract=off", "--expt-relaxed-constexpr", "-Xptxas", "-v"]


def nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def needs_build():
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    return any(os.path.getmtime(os.path.join(HERE, f)) > t for f in SOURCES + HEADERS + ["build.py"])


def build(force=False, verbose=False, out=None, extra=()):
    """out / extra: build an experimental variant next to the product library (select it with TR_LIB=path)."""
    global OUT
    if out:
        OUT, force = out, True
    if not force and not needs_build():
        return OUT
    objdir = os.path.join(HERE, "build" if not out else "build_" + os.path.basename(out))
    os.makedirs(objdir, exist_ok=True)
    objs = []
    procs = []
    for src in SOURCES:
        obj = os.path.join(objdir, src.replace(".cu", ".o"))
        objs.append(obj)
        cmd = [nvcc()] + NVCC_FLAGS + list(extra) + ["-c", os.path.join(HERE, src), "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    log = []
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        log.append(f"==== {src}\n{out}")
        if p.returncode != 0:
            failed = True
    with open(os.path.join(objdir, "ptxas.log"), "w") as f:
        f.write("\n".join(log))
    if failed or verbose:
        sys.stderr.write("\n".join(log))
    if failed:
        raise RuntimeError("nvcc failed (see output above)")
    link = [nvcc(), "-shared", "-o", OUT] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-ldl"]
    subprocess.check_call(link)
    return OUT


if __name__ == "__main__":
    extra = [a for a in sys.argv[1:] if a.startswith("-D")]
    out = next((a.split("=", 1)[1] for a in sys.argv[1:] if a.startswith("--out=")), None)
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv, out=out, extra=extra))
