// k_accel.cu — acceleration structures for the ray-queried shadows: host-side builders and the ray-batch kernel.
//
// Reference behaviour:
//   build_acceleration_structures_from_primitives        src/acceleration_structures.rs:6-104   (one per primitive)
//   build_top_level_acceleration_structure_from_instances                      :106-186  (instances, PREFER_FAST_TRACE)
//   update_top_level_acceleration_structure_from_instances                     :188-263  (after an instance moved)
//   the instance filter `draw_buffer_index < 2`           src/main.rs:614-625
// The reference hands both builds to the Vulkan driver; here they are binned-SAH builds on the host, run at load time
// and by tr_update_top_level_acceleration_structure, which reads the instances back and waits for the GPU.  When
// instances move every frame (the reference's --rotate-model), tr_update_top_level_acceleration_structure_async rebuilds
// the top level on the device in stream order instead (k_accel_device.cu), and tr_update_mesh_vertices refits the bottom
// level there from the parent links and triangle sources this build uploads (k_mesh_update.cu).  What the trees must
// guarantee is in tr_device_accel.cuh: inner boxes are exact unions and the depth of either level stays below kAccelStack.
#include <algorithm>
#include <cmath>
#include <cstring>
#include <limits>

#include "tr_device_accel.cuh"
#include "tr_internal.h"

using namespace trd;

namespace {

struct Box {
    float lo[3], hi[3];
};
inline Box box_empty() {
    const float inf = std::numeric_limits<float>::infinity();
    return Box{{inf, inf, inf}, {-inf, -inf, -inf}};
}
inline void box_grow(Box& b, const float* p) {
    for (int k = 0; k < 3; k++) {
        b.lo[k] = fminf(b.lo[k], p[k]);
        b.hi[k] = fmaxf(b.hi[k], p[k]);
    }
}
inline void box_union(Box& b, const Box& o) {
    box_grow(b, o.lo);
    box_grow(b, o.hi);
}
inline float box_area(const Box& b) {
    const float dx = b.hi[0] - b.lo[0], dy = b.hi[1] - b.lo[1], dz = b.hi[2] - b.lo[2];
    if (!(dx >= 0.0f)) return 0.0f;
    return dx * dy + dy * dz + dz * dx;
}

struct Item {
    Box box;
    uint32_t id;
};

constexpr int kBins = 16;
constexpr int kSahDepth = 28;  // below this depth every split halves the range, so depth <= 28 + log2(n) < kAccelStack

// Returns the child reference for items[first, first+count) and the exact union of their boxes.  Leaves refer to
// positions in the (reordered) item array.
int32_t build_range(std::vector<AccelNode>& nodes, std::vector<Item>& items, uint32_t first, uint32_t count, int depth,
                    uint32_t leaf_max, Box* out_box) {
    Box box = box_empty(), cbox = box_empty();
    for (uint32_t i = 0; i < count; i++) {
        const Box& b = items[first + i].box;
        box_union(box, b);
        const float c[3] = {b.lo[0] + b.hi[0], b.lo[1] + b.hi[1], b.lo[2] + b.hi[2]};
        box_grow(cbox, c);
    }
    *out_box = box;
    if (count <= leaf_max) return (int32_t) ~(first | ((count - 1u) << 28));

    // widest centroid axis: used by the median fallback
    int axis = 0;
    float ext = cbox.hi[0] - cbox.lo[0];
    for (int k = 1; k < 3; k++)
        if (cbox.hi[k] - cbox.lo[k] > ext) {
            ext = cbox.hi[k] - cbox.lo[k];
            axis = k;
        }
    uint32_t mid = 0;
    if (depth < kSahDepth && ext > 0.0f && count > 4u) {
        // binned surface-area heuristic, best split over the three axes
        float best = std::numeric_limits<float>::infinity();
        int best_axis = -1, best_split = -1;
        float best_scale = 0.0f;
        for (int ax = 0; ax < 3; ax++) {
            const float e = cbox.hi[ax] - cbox.lo[ax];
            if (!(e > 0.0f)) continue;
            uint32_t bin_n[kBins] = {};
            Box bin_b[kBins];
            for (int b = 0; b < kBins; b++) bin_b[b] = box_empty();
            const float scale = (float)kBins / e;
            for (uint32_t i = 0; i < count; i++) {
                const Item& it = items[first + i];
                int b = (int)(((it.box.lo[ax] + it.box.hi[ax]) - cbox.lo[ax]) * scale);
                b = b < 0 ? 0 : (b >= kBins ? kBins - 1 : b);
                bin_n[b]++;
                box_union(bin_b[b], it.box);
            }
            float right_area[kBins];
            uint32_t right_n[kBins];
            Box acc = box_empty();
            uint32_t n = 0;
            for (int b = kBins - 1; b > 0; b--) {
                box_union(acc, bin_b[b]);
                n += bin_n[b];
                right_area[b] = box_area(acc);
                right_n[b] = n;
            }
            acc = box_empty();
            n = 0;
            for (int b = 0; b < kBins - 1; b++) {
                box_union(acc, bin_b[b]);
                n += bin_n[b];
                if (n == 0 || right_n[b + 1] == 0) continue;
                const float cost = box_area(acc) * (float)n + right_area[b + 1] * (float)right_n[b + 1];
                if (cost < best) {
                    best = cost;
                    best_axis = ax;
                    best_split = b;
                    best_scale = scale;
                }
            }
        }
        if (best_axis >= 0) {
            const int ax = best_axis;
            auto it = std::partition(items.begin() + first, items.begin() + first + count, [&](const Item& x) {
                int b = (int)(((x.box.lo[ax] + x.box.hi[ax]) - cbox.lo[ax]) * best_scale);
                b = b < 0 ? 0 : (b >= kBins ? kBins - 1 : b);
                return b <= best_split;
            });
            mid = (uint32_t)(it - (items.begin() + first));
        }
    }
    if (mid == 0 || mid == count) {  // median split on the centroid (ties by id keep it deterministic)
        mid = count / 2;
        std::nth_element(items.begin() + first, items.begin() + first + mid, items.begin() + first + count,
                         [axis](const Item& x, const Item& y) {
                             const float cx = x.box.lo[axis] + x.box.hi[axis], cy = y.box.lo[axis] + y.box.hi[axis];
                             return cx < cy || (cx == cy && x.id < y.id);
                         });
    }
    const int32_t idx = (int32_t)nodes.size();
    nodes.push_back(AccelNode{});
    Box b0, b1;
    const int32_t c0 = build_range(nodes, items, first, mid, depth + 1, leaf_max, &b0);
    const int32_t c1 = build_range(nodes, items, first + mid, count - mid, depth + 1, leaf_max, &b1);
    AccelNode& n = nodes[idx];
    memcpy(n.lo0, b0.lo, 12);
    memcpy(n.hi0, b0.hi, 12);
    memcpy(n.lo1, b1.lo, 12);
    memcpy(n.hi1, b1.hi, 12);
    n.c0 = c0;
    n.c1 = c1;
    return idx;
}

// Appends a tree over `items` to `nodes`; returns the index of its root, which is always an inner node.
uint32_t build_tree(std::vector<AccelNode>& nodes, std::vector<Item>& items, uint32_t leaf_max) {
    const uint32_t root = (uint32_t)nodes.size();
    Box box;
    if (items.empty()) {  // nothing below: both children are boxes no ray can enter
        AccelNode n{};
        const Box e = box_empty();
        memcpy(n.lo0, e.lo, 12); memcpy(n.hi0, e.hi, 12); memcpy(n.lo1, e.lo, 12); memcpy(n.hi1, e.hi, 12);
        n.c0 = n.c1 = ~0;
        nodes.push_back(n);
        return root;
    }
    const int32_t c = build_range(nodes, items, 0, (uint32_t)items.size(), 0, leaf_max, &box);
    if (c < 0) {  // a single leaf: wrap it
        AccelNode n{};
        const Box e = box_empty();
        memcpy(n.lo0, box.lo, 12); memcpy(n.hi0, box.hi, 12); memcpy(n.lo1, e.lo, 12); memcpy(n.hi1, e.hi, 12);
        n.c0 = n.c1 = c;
        nodes.push_back(n);
    }
    return root;
}

// glam 0.19 scalar operation order (oracle/vecmath.h); the host compiler runs with -ffp-contract=off
struct H3 { float x, y, z; };
inline H3 h3(float x, float y, float z) { return H3{x, y, z}; }
inline float hdot(H3 a, H3 b) { return (a.x * b.x + a.y * b.y) + a.z * b.z; }
inline H3 hscale(H3 a, float s) { return h3(a.x * s, a.y * s, a.z * s); }
inline H3 hadd(H3 a, H3 b) { return h3(a.x + b.x, a.y + b.y, a.z + b.z); }
inline H3 hcross(H3 a, H3 b) { return h3(a.y * b.z - b.y * a.z, a.z * b.x - b.z * a.x, a.x * b.y - b.x * a.y); }
inline H3 hquat_mul(float qx, float qy, float qz, float qw, H3 v) {
    const H3 b = h3(qx, qy, qz);
    const float b2 = hdot(b, b);
    H3 r = hscale(v, qw * qw - b2);
    r = hadd(r, hscale(b, hdot(v, b) * 2.0f));
    r = hadd(r, hscale(hcross(b, v), qw * 2.0f));
    return r;
}

__global__ void __launch_bounds__(128) trace_rays_kernel(AccelDesc acc, uint32_t n, const float* __restrict__ origins,
                                                         const float* __restrict__ directions, const float* __restrict__ t_max,
                                                         uint8_t* __restrict__ lit) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const f3 o = mk3(origins[i * 3], origins[i * 3 + 1], origins[i * 3 + 2]);
    const f3 d = mk3(directions[i * 3], directions[i * 3 + 1], directions[i * 3 + 2]);
    lit[i] = accel_occluded(acc, o, d, t_max[i]) ? 0 : 1;
}

}  // namespace

namespace tr {

AccelDesc accel_desc(const tr_ctx* c) {
    AccelDesc a;
    a.tlas_nodes = c->accel_tlas.as<float4>();
    a.blas_nodes = c->accel_blas.as<float4>();
    a.instances = c->accel_inst.as<float4>();
    a.tris = c->accel_tris.as<float4>();
    a.n_instances = c->accel_n_instances;
    a.pad = 0;
    return a;
}

static int32_t upload_vec(tr_ctx* c, DevBuf& b, const void* src, size_t bytes) {
    TR_TRY(b.ensure(bytes ? bytes : 64));
    if (bytes) TR_CUDA(cudaMemcpyAsync(b.p, src, bytes, cudaMemcpyHostToDevice, c->stream));
    return TR_OK;
}

// top level: instances whose primitive draws into buffer 0 or 1, src/main.rs:614-625
int32_t accel_build_tlas(tr_ctx* c) {
    if (!c->accel_blas_valid) return fail(TR_ERR_STATE, "top-level build: bottom-level structures missing (tr_build_acceleration_structures)");
    std::vector<tr_instance> inst(c->n_instances);
    if (c->n_instances)
        TR_CUDA(cudaMemcpyAsync(inst.data(), c->instances.p, sizeof(tr_instance) * c->n_instances, cudaMemcpyDeviceToHost, c->stream));
    // the primitive boxes: the device table is their source of truth (a bottom-level refit rewrites them in stream order)
    std::vector<TlasPrim> prims(c->n_primitives);
    if (c->n_primitives)
        TR_CUDA(cudaMemcpyAsync(prims.data(), c->accel_prim_table.p, sizeof(TlasPrim) * c->n_primitives, cudaMemcpyDeviceToHost, c->stream));
    TR_CUDA(cudaStreamSynchronize(c->stream));
    std::vector<AccelInstance> records;
    std::vector<Item> items;
    for (uint32_t i = 0; i < c->n_instances; i++) {
        const uint32_t p = inst[i].primitive_id;
        if (p >= c->n_primitives) return fail(TR_ERR_INVALID_ARG, "top-level build: instance %u refers to primitive %u of %u", i, p, c->n_primitives);
        if (c->h_prim_bucket[p] >= 2u || c->h_prim_tris[p] == 0u) continue;
        const tr_packed_similarity& s = inst[i].transform;
        AccelInstance r{};
        r.tx = s.translation_and_scale.x; r.ty = s.translation_and_scale.y; r.tz = s.translation_and_scale.z;
        const float scale = s.translation_and_scale.w;
        r.inv_scale = 1.0f / scale;
        r.qx = -s.rotation.x; r.qy = -s.rotation.y; r.qz = -s.rotation.z; r.qw = s.rotation.w;
        Box w = box_empty();
        const float* lo = prims[p].lo;
        const float* hi = prims[p].hi;
        for (int k = 0; k < 8; k++) {  // Similarity * Vec3 (shared-structs lib.rs:216-220) on the eight corners
            const H3 corner = h3(k & 1 ? hi[0] : lo[0], k & 2 ? hi[1] : lo[1], k & 4 ? hi[2] : lo[2]);
            const H3 wp = hadd(h3(r.tx, r.ty, r.tz), hscale(hquat_mul(s.rotation.x, s.rotation.y, s.rotation.z, s.rotation.w, corner), scale));
            const float q[3] = {wp.x, wp.y, wp.z};
            box_grow(w, q);
        }
        memcpy(r.lo, w.lo, 12);
        memcpy(r.hi, w.hi, 12);
        r.blas_root = c->h_prim_root[p];
        r.tri_base = c->h_prim_tri_base[p];
        items.push_back(Item{w, (uint32_t)records.size()});
        records.push_back(r);
    }
    std::vector<AccelNode> nodes;
    build_tree(nodes, items, 1);
    std::vector<AccelInstance> ordered(records.size());
    for (size_t k = 0; k < items.size(); k++) ordered[k] = records[items[k].id];
    TR_TRY(upload_vec(c, c->accel_tlas, nodes.data(), nodes.size() * sizeof(AccelNode)));
    TR_TRY(upload_vec(c, c->accel_inst, ordered.data(), ordered.size() * sizeof(AccelInstance)));
    TR_CUDA(cudaStreamSynchronize(c->stream));  // the host vectors go away
    c->accel_n_instances = (uint32_t)ordered.size();
    c->accel_tlas_valid = true;
    return TR_OK;
}

int32_t accel_build(tr_ctx* c) {
    if (!c->n_vertices || !c->n_indices) return fail(TR_ERR_STATE, "tr_build_acceleration_structures: mesh not set");
    if (!c->n_primitives) return fail(TR_ERR_STATE, "tr_build_acceleration_structures: primitives not set");
    std::vector<float> pos((size_t)c->n_vertices * 3);
    std::vector<uint32_t> idx(c->n_indices);
    std::vector<tr_primitive_info> prims(c->n_primitives);
    TR_CUDA(cudaMemcpyAsync(pos.data(), c->mesh_pos.p, pos.size() * 4, cudaMemcpyDeviceToHost, c->stream));
    TR_CUDA(cudaMemcpyAsync(idx.data(), c->mesh_idx.p, idx.size() * 4, cudaMemcpyDeviceToHost, c->stream));
    TR_CUDA(cudaMemcpyAsync(prims.data(), c->primitives.p, prims.size() * sizeof(tr_primitive_info), cudaMemcpyDeviceToHost, c->stream));
    TR_CUDA(cudaStreamSynchronize(c->stream));

    std::vector<AccelNode> nodes;
    std::vector<float4> tris;
    std::vector<uint32_t> tri_src;                       // first index of every leaf-order triangle (the refit's gather)
    std::vector<TlasPrim> table(c->n_primitives);
    c->h_prim_root.assign(c->n_primitives, 0u);
    c->h_prim_tri_base.assign(c->n_primitives, 0u);
    c->h_prim_bucket.assign(c->n_primitives, 0u);
    std::vector<Item> items;
    for (uint32_t p = 0; p < c->n_primitives; p++) {  // one bottom-level structure per primitive, :47-52
        const tr_primitive_info& pr = prims[p];
        const uint32_t nt = pr.index_count / 3;
        if ((uint64_t)pr.first_index + pr.index_count > c->n_indices)
            return fail(TR_ERR_INVALID_ARG, "tr_build_acceleration_structures: primitive %u indexes past the index buffer", p);
        if (nt >= (1u << 28)) return fail(TR_ERR_UNSUPPORTED, "tr_build_acceleration_structures: primitive %u has %u triangles", p, nt);
        c->h_prim_bucket[p] = pr.draw_buffer_index;
        c->h_prim_tri_base[p] = (uint32_t)(tris.size() / 3);
        items.clear();
        items.reserve(nt);
        Box pb = box_empty();
        for (uint32_t t = 0; t < nt; t++) {
            Box b = box_empty();
            for (int k = 0; k < 3; k++) {
                const uint32_t v = idx[pr.first_index + t * 3 + k];
                if (v >= c->n_vertices) return fail(TR_ERR_INVALID_ARG, "tr_build_acceleration_structures: index %u past %u vertices", v, c->n_vertices);
                box_grow(b, &pos[(size_t)v * 3]);
            }
            box_union(pb, b);
            items.push_back(Item{b, t});
        }
        c->h_prim_root[p] = build_tree(nodes, items, 4);
        for (const Item& it : items) {  // triangles in leaf order
            tri_src.push_back(pr.first_index + it.id * 3);
            for (int k = 0; k < 3; k++) {
                const float* v = &pos[(size_t)idx[pr.first_index + it.id * 3 + k] * 3];
                tris.push_back(make_float4(v[0], v[1], v[2], 0.0f));
            }
        }
        memcpy(table[p].lo, pb.lo, 12);
        memcpy(table[p].hi, pb.hi, 12);
        table[p].blas_root = c->h_prim_root[p];
        table[p].tri_base = c->h_prim_tri_base[p];
        table[p].keep = pr.draw_buffer_index < 2u && nt != 0u;
    }
    // the refit's parent links: -1 at a root (build_tree appends every tree in preorder, children after their parent)
    std::vector<int32_t> parent(nodes.size(), -1);
    for (size_t i = 0; i < nodes.size(); i++)
        for (int32_t ch : {nodes[i].c0, nodes[i].c1})
            if (ch >= 0) parent[ch] = (int32_t)i;
    if (c->h_prim_tris.size() != c->n_primitives) {
        c->h_prim_tris.resize(c->n_primitives);
        for (uint32_t p = 0; p < c->n_primitives; p++) c->h_prim_tris[p] = prims[p].index_count / 3;
    }
    TR_TRY(upload_vec(c, c->accel_blas, nodes.data(), nodes.size() * sizeof(AccelNode)));
    TR_TRY(upload_vec(c, c->accel_tris, tris.data(), tris.size() * sizeof(float4)));
    TR_TRY(upload_vec(c, c->accel_prim_table, table.data(), table.size() * sizeof(TlasPrim)));
    // refit tables (k_mesh_update.cu): parents [nodes], arrival counters [nodes], triangle sources [triangles]
    const size_t nn = nodes.size(), nt = tri_src.size();
    TR_TRY(c->accel_refit.ensure((nn * 2 + nt) * 4));
    TR_CUDA(cudaMemcpyAsync(c->accel_refit.p, parent.data(), nn * 4, cudaMemcpyHostToDevice, c->stream));
    if (nt) TR_CUDA(cudaMemcpyAsync(c->accel_refit.as<uint32_t>() + nn * 2, tri_src.data(), nt * 4, cudaMemcpyHostToDevice, c->stream));
    TR_CUDA(cudaStreamSynchronize(c->stream));
    c->accel_blas_nodes = (uint32_t)nn;
    c->accel_n_tris = (uint32_t)nt;
    c->accel_blas_valid = true;
    return accel_build_tlas(c);
}

int32_t launch_trace_rays(tr_ctx* c, uint32_t n, const float* d_origins, const float* d_directions, const float* d_t_max, uint8_t* d_lit) {
    if (!n) return TR_OK;
    trace_rays_kernel<<<(n + 127) / 128, 128, 0, c->stream>>>(accel_desc(c), n, d_origins, d_directions, d_t_max, d_lit);
    count_launches(1);
    TR_CUDA(cudaGetLastError());
    return TR_OK;
}

}  // namespace tr
