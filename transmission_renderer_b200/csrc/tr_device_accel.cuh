// tr_device_accel.cuh — ray-queried shadows: acceleration-structure layout and the any-hit traversal (sm_100a).
//
// Reference behaviour: trace_shadow_ray (shader/src/lighting.rs:97-125) against the top-level structure of
// src/acceleration_structures.rs (one bottom-level structure per primitive, instances with draw_buffer_index < 2,
// src/main.rs:614-625).  B200 has no ray-tracing units, so the query is a software walk of two-level bounding-volume
// hierarchies.  The RESULT is defined independently of the trees (DESIGN.md "Ray-queried shadows", oracle/shadow.c):
//
//   occluded(ray) := exists instance i:  slab(world ray, world_box_i)  and  exists triangle k of its primitive:
//                    slab(object ray_i, box_k)  and  hit64(object ray_i, triangle k)
//
// slab() is monotone in the box, every inner box of the trees is the exact union of what is below it, so skipping a
// subtree whose box fails can never change the outcome.  All of it runs in the exact regime (unfused IEEE operations
// in a fixed order): the outcome is a bit, and it has to be the oracle's bit.
#pragma once

#include "tr_device_math.cuh"

namespace trd {

struct AccelNode {  // 64 B: an inner node carries the boxes of its two children
    float lo0[3], hi0[3], lo1[3], hi1[3];
    int32_t c0, c1;  // >= 0: inner node (index into the same array); < 0: leaf, ~c = first | (count - 1) << 28
    uint32_t pad[2];
};
static_assert(sizeof(AccelNode) == 64, "AccelNode");

struct AccelInstance {  // 64 B, stored in top-level leaf order
    float tx, ty, tz, inv_scale;  // Similarity translation, 1 / scale
    float qx, qy, qz, qw;         // conjugate of the Similarity rotation
    float lo[3], hi[3];           // world box (the eight corners of the primitive's box through the Similarity)
    uint32_t blas_root;           // root node of the primitive's tree in blas_nodes
    uint32_t tri_base;            // first triangle of the primitive in tris
};
static_assert(sizeof(AccelInstance) == 64, "AccelInstance");

struct TlasPrim {  // what the top level needs of a primitive: the per-primitive table on the device (k_accel_device.cu)
    float lo[3], hi[3];       // object-space box; a bottom-level refit rewrites it (k_mesh_update.cu)
    uint32_t blas_root, tri_base;
    uint32_t keep;            // draw_buffer_index < 2 and at least one triangle (src/main.rs:614-625)
    uint32_t pad[3];
};
static_assert(sizeof(TlasPrim) == 48, "TlasPrim");

struct AccelDesc {
    const float4* tlas_nodes;  // AccelNode[]; node 0 is the root
    const float4* blas_nodes;  // AccelNode[] of all primitives
    const float4* instances;   // AccelInstance[]
    const float4* tris;        // three float4 per triangle (v0, v1, v2; w unused), bottom-level leaf order per primitive
    uint32_t n_instances;      // 0: nothing can occlude
    uint32_t pad;
};

constexpr float kShadowTMin = 0.001f;      // lighting.rs:109
constexpr float kSunTMax = 10000.0f;       // lighting.rs:31, 163
// Traversal stack.  A push onto a full stack is dropped (sp < kAccelStack), which would lose a subtree and give a wrong bit,
// not an error, so every builder bounds the depth of its trees below it:
//   k_accel.cu (host, both levels): median splits below depth 28, so depth <= 28 + log2(n) < 64.
//   k_accel_device.cu (device, top level): a radix tree over keys (30-bit Morton code, position); positions break ties, so
//   the keys are distinct 54-bit strings (tr_set_instances keeps n below 2^24).  Every inner node splits its range at the
//   first bit where its keys differ, so a child's common prefix is strictly longer than its parent's; the prefixes run
//   from 0 to 53 bits, so a root-to-leaf path has at most 54 inner nodes and the depth is <= 55 < 64
//   (tests/test_gpu_accel_update.py checks it on equal codes, geometric chains and wide scale ranges).
//   k_accel_build.cu (device, bottom level): H-PLOC has no depth bound of its own, so the build measures every primitive's
//   depth and builds a primitive deeper than kAccelStack - 1 again as the plain radix tree over the keys (30-bit Morton
//   code, position within the primitive); positions are below 2^28, so the keys are distinct 58-bit strings, every inner
//   node splits at the first bit where its keys differ, the prefixes run from 0 to 57 bits, and the depth is <= 59 < 64
//   (tests/test_gpu_accel_build.py checks it, with the fallback forced on ordinary meshes and on pathological ones).
constexpr int kAccelStack = 64;

struct AccelRay {
    float o[3], d[3], inv[3];
    float t_min, t_max;
};

TRD AccelRay make_accel_ray(f3 o, f3 d, float t_min, float t_max) {
    AccelRay r;
    r.o[0] = o.x; r.o[1] = o.y; r.o[2] = o.z;
    r.d[0] = d.x; r.d[1] = d.y; r.d[2] = d.z;
    r.inv[0] = xdiv(1.0f, d.x); r.inv[1] = xdiv(1.0f, d.y); r.inv[2] = xdiv(1.0f, d.z);
    r.t_min = t_min;
    r.t_max = t_max;
    return r;
}

// the fp32 interval test of the definition; fmaxf / fminf drop a NaN operand (0 * inf) like the oracle's
TRD bool accel_slab(const AccelRay& r, float lox, float loy, float loz, float hix, float hiy, float hiz) {
    float tn = r.t_min, tf = r.t_max;
    {
        const bool neg = r.inv[0] < 0.0f;
        tn = fmaxf(tn, xmul(xsub(neg ? hix : lox, r.o[0]), r.inv[0]));
        tf = fminf(tf, xmul(xsub(neg ? lox : hix, r.o[0]), r.inv[0]));
    }
    {
        const bool neg = r.inv[1] < 0.0f;
        tn = fmaxf(tn, xmul(xsub(neg ? hiy : loy, r.o[1]), r.inv[1]));
        tf = fminf(tf, xmul(xsub(neg ? loy : hiy, r.o[1]), r.inv[1]));
    }
    {
        const bool neg = r.inv[2] < 0.0f;
        tn = fmaxf(tn, xmul(xsub(neg ? hiz : loz, r.o[2]), r.inv[2]));
        tf = fminf(tf, xmul(xsub(neg ? loz : hiz, r.o[2]), r.inv[2]));
    }
    return tn <= xmul(tf, 1.00000024f);  // 1 + 2^-22
}

// Moeller-Trumbore in double on the fp32 inputs, both faces, t_min < t < t_max (oracle/shadow.c hit64)
TRD bool accel_hit64(const AccelRay& r, float4 a, float4 b, float4 c) {
    const double v0[3] = {(double)a.x, (double)a.y, (double)a.z};
    const double e1[3] = {__dsub_rn((double)b.x, v0[0]), __dsub_rn((double)b.y, v0[1]), __dsub_rn((double)b.z, v0[2])};
    const double e2[3] = {__dsub_rn((double)c.x, v0[0]), __dsub_rn((double)c.y, v0[1]), __dsub_rn((double)c.z, v0[2])};
    const double tv[3] = {__dsub_rn((double)r.o[0], v0[0]), __dsub_rn((double)r.o[1], v0[1]), __dsub_rn((double)r.o[2], v0[2])};
    const double d[3] = {(double)r.d[0], (double)r.d[1], (double)r.d[2]};
    auto cross = [](const double* x, const double* y, double* out) {
        out[0] = __dsub_rn(__dmul_rn(x[1], y[2]), __dmul_rn(x[2], y[1]));
        out[1] = __dsub_rn(__dmul_rn(x[2], y[0]), __dmul_rn(x[0], y[2]));
        out[2] = __dsub_rn(__dmul_rn(x[0], y[1]), __dmul_rn(x[1], y[0]));
    };
    auto dot = [](const double* x, const double* y) {
        return __dadd_rn(__dadd_rn(__dmul_rn(x[0], y[0]), __dmul_rn(x[1], y[1])), __dmul_rn(x[2], y[2]));
    };
    double p[3], q[3];
    cross(d, e2, p);
    const double det = dot(e1, p);
    if (det == 0.0) return false;
    const double inv = __ddiv_rn(1.0, det);
    const double u = __dmul_rn(dot(tv, p), inv);
    if (!(u >= 0.0 && u <= 1.0)) return false;
    cross(tv, e1, q);
    const double w = __dmul_rn(dot(d, q), inv);
    if (!(w >= 0.0 && __dadd_rn(u, w) <= 1.0)) return false;
    const double t = __dmul_rn(dot(e2, q), inv);
    return t > (double)r.t_min && t < (double)r.t_max;
}

TRD bool accel_instance_occludes(const AccelDesc& acc, const float4* inst, f3 o, f3 d, float t_min, float t_max) {
    const float4 i0 = __ldg(inst), i1 = __ldg(inst + 1), i3 = __ldg(inst + 3);
    // object ray: o' = (conj(q) * (o - t)) / s, d' = (conj(q) * d) / s, so t keeps its world meaning
    const f3 oo = xscale3(xquat_mul3(i1.x, i1.y, i1.z, i1.w, xsub3(o, mk3(i0.x, i0.y, i0.z))), i0.w);
    const f3 od = xscale3(xquat_mul3(i1.x, i1.y, i1.z, i1.w, d), i0.w);
    const AccelRay r = make_accel_ray(oo, od, t_min, t_max);
    const uint32_t tri_base = __float_as_uint(i3.w);
    int32_t stack[kAccelStack];
    int sp = 0;
    int32_t node = (int32_t)__float_as_uint(i3.z);
    while (true) {
        const float4* n = acc.blas_nodes + (size_t)node * 4;
        const float4 n0 = __ldg(n), n1 = __ldg(n + 1), n2 = __ldg(n + 2), n3 = __ldg(n + 3);
        const bool h0 = accel_slab(r, n0.x, n0.y, n0.z, n0.w, n1.x, n1.y);
        const bool h1 = accel_slab(r, n1.z, n1.w, n2.x, n2.y, n2.z, n2.w);
        const int32_t c[2] = {__float_as_int(n3.x), __float_as_int(n3.y)};
        const bool h[2] = {h0, h1};
        int32_t next = -1;
        bool have_next = false;
#pragma unroll
        for (int k = 0; k < 2; k++) {
            if (!h[k]) continue;
            if (c[k] < 0) {  // leaf: the triangle's own box, then the double-precision test
                const uint32_t code = ~(uint32_t)c[k];
                const uint32_t first = code & 0x0fffffffu, count = (code >> 28) + 1u;
                for (uint32_t j = 0; j < count; j++) {
                    const float4* tp = acc.tris + (size_t)(tri_base + first + j) * 3;
                    const float4 a = __ldg(tp), b = __ldg(tp + 1), cc = __ldg(tp + 2);
                    if (accel_slab(r, fminf(fminf(a.x, b.x), cc.x), fminf(fminf(a.y, b.y), cc.y), fminf(fminf(a.z, b.z), cc.z),
                                   fmaxf(fmaxf(a.x, b.x), cc.x), fmaxf(fmaxf(a.y, b.y), cc.y), fmaxf(fmaxf(a.z, b.z), cc.z)) &&
                        accel_hit64(r, a, b, cc))
                        return true;
                }
            } else if (!have_next) {
                next = c[k];
                have_next = true;
            } else if (sp < kAccelStack) {
                stack[sp++] = c[k];
            }
        }
        if (have_next) {
            node = next;
        } else {
            if (sp == 0) return false;
            node = stack[--sp];
        }
    }
}

// trace_shadow_ray, lighting.rs:97-125: true = some geometry between t_min and t_max
TRD bool accel_occluded(const AccelDesc& acc, f3 o, f3 d, float t_max) {
    if (acc.n_instances == 0u) return false;
    const AccelRay r = make_accel_ray(o, d, kShadowTMin, t_max);
    int32_t stack[kAccelStack];
    int sp = 0;
    int32_t node = 0;
    while (true) {
        const float4* n = acc.tlas_nodes + (size_t)node * 4;
        const float4 n0 = __ldg(n), n1 = __ldg(n + 1), n2 = __ldg(n + 2), n3 = __ldg(n + 3);
        const bool h0 = accel_slab(r, n0.x, n0.y, n0.z, n0.w, n1.x, n1.y);
        const bool h1 = accel_slab(r, n1.z, n1.w, n2.x, n2.y, n2.z, n2.w);
        const int32_t c[2] = {__float_as_int(n3.x), __float_as_int(n3.y)};
        const bool h[2] = {h0, h1};
        int32_t next = -1;
        bool have_next = false;
#pragma unroll
        for (int k = 0; k < 2; k++) {
            if (!h[k]) continue;
            if (c[k] < 0) {  // leaf: instances; the world box is part of the definition, so it is tested on its own
                const uint32_t code = ~(uint32_t)c[k];
                const uint32_t first = code & 0x0fffffffu, count = (code >> 28) + 1u;
                for (uint32_t j = 0; j < count; j++) {
                    const float4* inst = acc.instances + (size_t)(first + j) * 4;
                    const float4 b0 = __ldg(inst + 2), b1 = __ldg(inst + 3);
                    if (accel_slab(r, b0.x, b0.y, b0.z, b0.w, b1.x, b1.y) &&
                        accel_instance_occludes(acc, inst, o, d, kShadowTMin, t_max))
                        return true;
                }
            } else if (!have_next) {
                next = c[k];
                have_next = true;
            } else if (sp < kAccelStack) {
                stack[sp++] = c[k];
            }
        }
        if (have_next) {
            node = next;
        } else {
            if (sp == 0) return false;
            node = stack[--sp];
        }
    }
}

}  // namespace trd
