"""examples/frame_group.c is a C11 host of the group entry points (tr_group_*): it compiles against the header with warnings as
errors, links libtr.so, and without a CUDA device fails loudly in the first call instead of falling back to anything."""
import os
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_group_c_host_compiles_and_fails_loudly_without_a_device(tmp_path):
    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    libdir = os.path.join(ROOT, "transmission_renderer_b200")
    exe = str(tmp_path / "frame_group")
    subprocess.check_call(["gcc", "-std=c11", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "examples", "frame_group.c"), "-L", libdir, "-ltr", f"-Wl,-rpath,{libdir}", "-lm",
                           "-o", exe])
    p = subprocess.run([exe], capture_output=True, text=True, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""), timeout=120)
    assert p.returncode == 3 and "tr_create" in p.stderr and "no CPU path" in p.stderr, (p.returncode, p.stdout, p.stderr)


def test_cpp_renderer_group_compiles_and_throws_without_a_device(tmp_path):
    """tr::RendererGroup (include/tr_host.hpp) builds against the library; without a device its constructor throws tr::Error."""
    if shutil.which("g++") is None:
        pytest.skip("no g++")
    src = tmp_path / "group.cpp"
    src.write_text('#include <cstdio>\n#include "tr_host.hpp"\n'
                   "int main() {\n"
                   "    try {\n"
                   "        tr::RendererGroup g({0, 0}, 64, 32);\n"
                   "        g.frame(tr_frame_params{});\n"
                   "        return g.read_srgb8().size() == 64 * 32 * 4 ? 0 : 1;\n"
                   "    } catch (const tr::Error& e) {\n"
                   '        std::fprintf(stderr, "%s\\n", e.what());\n'
                   "        return e.status() == TR_ERR_CUDA ? 3 : 4;\n"
                   "    }\n"
                   "}\n")
    libdir = os.path.join(ROOT, "transmission_renderer_b200")
    exe = str(tmp_path / "group")
    subprocess.check_call(["g++", "-std=c++17", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-L", libdir, "-ltr",
                           f"-Wl,-rpath,{libdir}", "-o", exe])
    p = subprocess.run([exe], capture_output=True, text=True, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""), timeout=120)
    assert p.returncode == 3 and "no CPU path" in p.stderr, (p.returncode, p.stderr)
