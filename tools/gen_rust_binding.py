"""Generates examples/tr_sys.rs — the COMPLETE Rust binding of include/tr_abi.h (every export, every ABI-own struct,
the status codes and flags) — from the header itself, so the binding a maintainer of the reference adds (INTEGRATION.md 1
shows its essential part by hand) cannot drift from the C ABI.

    python tools/gen_rust_binding.py            # rewrites examples/tr_sys.rs
    python tools/gen_rust_binding.py --check    # exit 1 if the file on disk differs

The shared-structs types are the reference's own (`shared_structs::Instance` ...): the header's copies of them are pinned to
the same bytes (static asserts + tests/test_abi_layout.py), so the Rust side passes its values by pointer unchanged.  No Rust
toolchain exists in this environment: the file is checked for completeness and consistency by tests/test_rust_binding.py,
not compiled.
"""
import os
import re
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "tr_abi.h")
OUT = os.path.join(ROOT, "examples", "tr_sys.rs")

SCALARS = {"int32_t": "i32", "uint32_t": "u32", "uint64_t": "u64", "int64_t": "i64", "uint16_t": "u16", "uint8_t": "u8", "size_t": "usize",
           "float": "f32", "double": "f64", "void": "std::os::raw::c_void", "char": "std::os::raw::c_char", "int": "std::os::raw::c_int"}
# the header's byte-for-byte copies of reference types -> the reference's own Rust types
REFERENCE_TYPES = {
    "tr_instance": "shared_structs::Instance", "tr_primitive_info": "shared_structs::PrimitiveInfo",
    "tr_material_info": "shared_structs::MaterialInfo", "tr_light": "shared_structs::Light", "tr_uniforms": "shared_structs::Uniforms",
    "tr_push_constants": "shared_structs::PushConstants", "tr_culling_push_constants": "shared_structs::CullingPushConstants",
    "tr_write_cluster_data_push_constants": "shared_structs::WriteClusterDataPushConstants",
    "tr_assign_lights_push_constants": "shared_structs::AssignLightsPushConstants", "tr_cluster_aabb": "shared_structs::ClusterAabb",
    "tr_baked_lottes_tonemapper_params": "colstodian::tonemap::BakedLottesTonemapperParams",   # what the host passes, src/main.rs:506,1547
    "tr_draw_indexed_indirect_command": "ash::vk::DrawIndexedIndirectCommand",
    "tr_mat4": "glam::Mat4", "tr_vec4": "glam::Vec4", "tr_quat": "glam::Quat", "tr_vec3a": "glam::Vec3A",
    "tr_vec2": "glam::Vec2", "tr_uvec2": "glam::UVec2", "tr_vec3": "[f32; 3]",   # glam::Vec3 is 12 bytes, align 4, like [f32; 3]
    "tr_light_cluster_coefficients": "shared_structs::LightClusterCoefficients", "tr_textures": "shared_structs::Textures",
    "tr_packed_similarity": "shared_structs::PackedSimilarity",
}
# opaque handles: only ever behind a pointer
OPAQUE = {"tr_ctx": "one per GPU / host thread", "tr_group": "contexts of one host thread rendering the bands of one frame"}
# ABI-own structs: generated as #[repr(C)] below
OWN_STRUCTS = ["tr_material_params", "tr_basic_brdf_params", "tr_brdf_result", "tr_transmission_btdf_params",
               "tr_ibl_volume_refraction_params", "tr_point_light_params", "tr_point_light_result", "tr_config", "tr_gbuffer_planes",
               "tr_gbuffer_planes_out", "tr_frame_params", "tr_frame_times"]


def camel(name):
    return "".join(p.capitalize() for p in name.split("_"))


def strip_comments(text):
    text = re.sub(r"/\*.*?\*/", " ", text, flags=re.S)
    return re.sub(r"//[^\n]*", " ", text)


def rust_type(ctype):
    """`const tr_instance*` -> `*const shared_structs::Instance`, `uint8_t* const*` -> `*const *mut u8` ..."""
    t = ctype.strip()
    if t.endswith("*"):
        inner = t[:-1].strip()
        ptr_const = False
        if inner.endswith("const"):          # `T* const*`: the pointer being pointed to is const
            inner, ptr_const = inner[:-5].strip(), True
        if inner.endswith("*"):              # pointer to pointer
            return ("*const " if ptr_const else "*mut ") + rust_type(inner)
        if inner.startswith("const "):
            return "*const " + rust_type(inner[6:])
        return "*mut " + rust_type(inner)
    if t.startswith("const "):
        t = t[6:].strip()
    if t in SCALARS:
        return SCALARS[t]
    if t in REFERENCE_TYPES:
        return REFERENCE_TYPES[t]
    if t in OPAQUE or t in OWN_STRUCTS:
        return camel(t)
    raise ValueError(f"unmapped C type {ctype!r}")


def parse_param(p):
    """-> (name, rust type).  Arrays (`uint8_t id[128]`, `uint64_t out[4]`) decay to pointers as in C."""
    p = p.strip()
    m = re.match(r"^(.*?)(\w+)\s*\[\s*\w*\s*\]$", p)
    if m:
        base, name = m.group(1).strip(), m.group(2)
        return name, ("*const " + rust_type(base[6:]) if base.startswith("const ") else "*mut " + rust_type(base))
    m = re.match(r"^(.*?)(\w+)$", p)
    return m.group(2), rust_type(m.group(1))


def parse_header(text):
    clean = strip_comments(text)
    defines = [(k, v) for k, v in re.findall(r"#define\s+(TR_(?:FLAG|FRAME|MAX|NUM|NCCL|IPC)\w*)\s+(\d+)u?\b", clean)]
    clean = "\n".join(l for l in clean.splitlines() if not l.lstrip().startswith("#"))   # preprocessor lines are not declarations
    fns = []
    for m in re.finditer(r"TR_API\s+(.*?)\b(tr_\w+)\s*\((.*?)\)\s*;", clean, flags=re.S):
        ret, name, params = m.group(1).strip(), m.group(2), " ".join(m.group(3).split())
        args = [] if params in ("", "void") else [parse_param(p) for p in params.split(",")]
        fns.append((name, args, rust_type(ret) if ret != "void" else None))
    structs = {}
    for m in re.finditer(r"typedef\s+struct\s*(?:TR_ALIGN16\s*)?\{(.*?)\}\s*(tr_\w+)\s*;", clean, flags=re.S):
        body, name = m.group(1), m.group(2)
        fields = []
        for decl in body.split(";"):
            decl = " ".join(decl.split())
            if not decl:
                continue
            first, *rest = [d.strip() for d in decl.split(",")]
            fname, ftype = parse_param(first)
            base = re.match(r"^(.*?)(\w+)(\s*\[.*\])?$", first).group(1)
            fields.append((fname, ftype))
            for r in rest:                       # `float a, b, c;` / `uint32_t width, height;`
                n, t = parse_param(base + " " + r)
                fields.append((n, t))
        structs[name] = fields
    enums = [(k, int(v)) for k, v in re.findall(r"\b(TR_(?:OK|ERR_\w+|LAYER_\w+|BUF_\w+))\s*=\s*(-?\d+)", clean)]
    return fns, structs, enums, defines


def generate():
    fns, structs, enums, defines = parse_header(open(HEADER).read())
    out = ["// examples/tr_sys.rs — GENERATED by tools/gen_rust_binding.py from include/tr_abi.h; do not edit.",
           "//",
           "// The complete raw FFI of libtr.so for the reference (a Rust application): drop it in as src/tr_sys.rs and link with",
           "// `cargo:rustc-link-lib=dylib=tr`.  The shared-structs / glam / ash types are the reference's own — the C header's copies of them",
           "// are pinned to the same bytes — so values are passed by pointer without conversion.  INTEGRATION.md maps every call onto the",
           "// place in src/main.rs it replaces.",
           "#![allow(non_camel_case_types, dead_code)]", ""]
    for name, what in OPAQUE.items():
        out.append(f"#[repr(C)] pub struct {camel(name)} {{ _private: [u8; 0] }}   // opaque: {what}")
    out.append("")
    for name in OWN_STRUCTS:
        fields = structs[name]
        out.append("#[repr(C)]")
        out.append("#[derive(Clone, Copy)]")
        out.append(f"pub struct {camel(name)} {{")
        for fname, ftype in fields:
            out.append(f"    pub {fname}: {ftype},")
        out.append("}")
        out.append("")
    for k, v in enums:
        out.append(f"pub const {k}: i32 = {v};")
    for k, v in defines:
        out.append(f"pub const {k}: u32 = {v};")
    out.append("")
    out.append('extern "C" {')
    for name, args, ret in fns:
        a = ", ".join(f"{n}: {t}" for n, t in args)
        out.append(f"    pub fn {name}({a})" + (f" -> {ret};" if ret else ";"))
    out.append("}")
    out.append("")
    out.append("/// Every non-zero status becomes an error carrying tr_last_error(): the reference propagates `anyhow::Result` with `?`")
    out.append("/// (src/main.rs:93) and logs-and-continues in the frame loop (:1453-1455).")
    out.append("pub fn check(status: i32) -> anyhow::Result<()> {")
    out.append("    if status == TR_OK { return Ok(()); }")
    out.append("    let msg = unsafe { std::ffi::CStr::from_ptr(tr_last_error()) }.to_string_lossy().into_owned();")
    out.append('    Err(anyhow::anyhow!("libtr status {}: {}", status, msg))')
    out.append("}")
    return "\n".join(out) + "\n"


if __name__ == "__main__":
    text = generate()
    if "--check" in sys.argv:
        sys.exit(0 if os.path.exists(OUT) and open(OUT).read() == text else 1)
    with open(OUT, "w") as f:
        f.write(text)
    print(OUT)
