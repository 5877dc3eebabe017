// k_accel_device.cu — the top-level acceleration structure rebuilt on the device, in stream order
// (tr_update_top_level_acceleration_structure_async).
//
// Reference behaviour: update_top_level_acceleration_structure_from_instances (src/acceleration_structures.rs:188-263),
// called after every instance write (src/main.rs:1263-1345), i.e. every frame under --rotate-model.  The host builder
// (k_accel.cu accel_build_tlas) reads the instances back and waits for the GPU; this one reads the instance buffer as
// the context's stream sees it and never waits.  It builds a linear BVH (Karras 2012, "Maximizing parallelism in the
// construction of BVHs, octrees, and k-d trees"): Morton codes of the world-box centroids, a stable radix sort, one
// radix-tree node per thread, boxes bottom-up.  The tree differs from the binned-SAH one, the occlusion result does not:
// the instance records are the host's byte for byte (same operation order, unfused), and every inner box is the exact
// union of its subtree (tr_device_accel.cuh).
//
// Launches per update (kAsyncTlasLaunches, fixed whatever the instance count): count, scan, records, bounds, codes,
// 4 x (histogram, scan, scatter), hierarchy, boxes = 19.
#include "tr_device_build.cuh"
#include "tr_internal.h"

using namespace trd;

namespace {

constexpr int kRadixPasses = 4;        // 30-bit codes in 8-bit digits

__device__ __forceinline__ uint32_t keep_of(const tr_instance* inst, const TlasPrim* prims, uint32_t i) {
    return prims[inst[i].primitive_id].keep;
}

// kept instances per block of kTile instances
__global__ void __launch_bounds__(kTile) tlas_count_kernel(const tr_instance* __restrict__ inst, uint32_t n,
                                                           const TlasPrim* __restrict__ prims, uint32_t* __restrict__ block_count) {
    const uint32_t i = blockIdx.x * kTile + threadIdx.x;
    const uint32_t k = i < n ? keep_of(inst, prims, i) : 0u;
    const int total = __syncthreads_count(k);
    if (threadIdx.x == 0) block_count[blockIdx.x] = (uint32_t)total;
}

// in-place exclusive prefix sum of data[0, len) by one block, kScanThreads entries at a time
__global__ void __launch_bounds__(kScanThreads) tlas_scan_kernel(uint32_t* __restrict__ data, uint32_t len) {
    __shared__ uint32_t warp_sum[32];
    uint32_t carry = 0;   // the sum of the entries before base
    for (uint32_t base = 0; base < len; base += kScanThreads) {
        const uint32_t i = base + threadIdx.x;
        uint32_t total;
        const uint32_t excl = carry + block_scan(i < len ? data[i] : 0u, warp_sum, &total);
        if (i < len) data[i] = excl;
        carry += total;
        __syncthreads();
    }
}

// The kept instances in instance order, and their AccelInstance records: k_accel.cu accel_build_tlas in the same exact
// operation order (the world box is part of the occlusion definition).
__global__ void __launch_bounds__(kTile) tlas_records_kernel(const tr_instance* __restrict__ inst, uint32_t n,
                                                             const TlasPrim* __restrict__ prims, const uint32_t* __restrict__ block_offset,
                                                             AccelInstance* __restrict__ rec) {
    __shared__ uint32_t warp_count[kTile / 32];
    const uint32_t i = blockIdx.x * kTile + threadIdx.x;
    const uint32_t k = i < n ? keep_of(inst, prims, i) : 0u;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t ballot = __ballot_sync(0xffffffffu, k);
    if (lane == 0) warp_count[warp] = __popc(ballot);
    __syncthreads();
    if (!k) return;
    uint32_t slot = block_offset[blockIdx.x] + __popc(ballot & ((1u << lane) - 1u));
    for (int w = 0; w < warp; w++) slot += warp_count[w];

    const tr_instance& in = inst[i];
    const TlasPrim& p = prims[in.primitive_id];
    const tr_vec4 ts = in.transform.translation_and_scale;
    const tr_quat q = in.transform.rotation;
    AccelInstance r;
    r.tx = ts.x; r.ty = ts.y; r.tz = ts.z;
    r.inv_scale = xdiv(1.0f, ts.w);
    r.qx = -q.x; r.qy = -q.y; r.qz = -q.z; r.qw = q.w;
    const float inf = __int_as_float(0x7f800000);
    float lo[3] = {inf, inf, inf}, hi[3] = {-inf, -inf, -inf};
#pragma unroll
    for (int c = 0; c < 8; c++) {  // Similarity * Vec3 (shared-structs lib.rs:216-220) on the eight corners
        const f3 corner = mk3(c & 1 ? p.hi[0] : p.lo[0], c & 2 ? p.hi[1] : p.lo[1], c & 4 ? p.hi[2] : p.lo[2]);
        const f3 wp = xadd3(mk3(r.tx, r.ty, r.tz), xscale3(xquat_mul3(q.x, q.y, q.z, q.w, corner), ts.w));
        lo[0] = fminf(lo[0], wp.x); hi[0] = fmaxf(hi[0], wp.x);
        lo[1] = fminf(lo[1], wp.y); hi[1] = fmaxf(hi[1], wp.y);
        lo[2] = fminf(lo[2], wp.z); hi[2] = fmaxf(hi[2], wp.z);
    }
    r.lo[0] = lo[0]; r.lo[1] = lo[1]; r.lo[2] = lo[2];
    r.hi[0] = hi[0]; r.hi[1] = hi[1]; r.hi[2] = hi[2];
    r.blas_root = p.blas_root;
    r.tri_base = p.tri_base;
    rec[slot] = r;
}

__device__ __forceinline__ float centroid(const AccelInstance& r, int k) { return r.lo[k] + r.hi[k]; }  // as build_range

// bounds of the centroids (lo + hi, as the host builder) by one block: out[0..2] lo, out[3..5] hi
__global__ void __launch_bounds__(kScanThreads) tlas_bounds_kernel(const AccelInstance* __restrict__ rec, uint32_t m,
                                                                   float* __restrict__ out) {
    __shared__ float s[6][kScanThreads / 32];
    const float inf = __int_as_float(0x7f800000);
    float v[6] = {inf, inf, inf, -inf, -inf, -inf};
    for (uint32_t i = threadIdx.x; i < m; i += kScanThreads) {
        const AccelInstance& r = rec[i];
        for (int k = 0; k < 3; k++) {
            const float c = centroid(r, k);
            v[k] = fminf(v[k], c);
            v[k + 3] = fmaxf(v[k + 3], c);
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1)
        for (int k = 0; k < 6; k++) {
            const float y = __shfl_xor_sync(0xffffffffu, v[k], o);
            v[k] = k < 3 ? fminf(v[k], y) : fmaxf(v[k], y);
        }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0)
        for (int k = 0; k < 6; k++) s[k][warp] = v[k];
    __syncthreads();
    if (threadIdx.x < 6) {
        const int k = threadIdx.x;
        float a = s[k][0];
        for (int w = 1; w < kScanThreads / 32; w++) a = k < 3 ? fminf(a, s[k][w]) : fmaxf(a, s[k][w]);
        out[k] = a;
    }
}

__global__ void __launch_bounds__(kTile) tlas_codes_kernel(const AccelInstance* __restrict__ rec, uint32_t m, const float* __restrict__ bounds,
                                                           uint32_t* __restrict__ keys, uint32_t* __restrict__ vals) {
    const uint32_t i = blockIdx.x * kTile + threadIdx.x;
    if (i >= m) return;
    const AccelInstance& r = rec[i];
    uint32_t code = 0;
    for (int k = 0; k < 3; k++) {
        const float ext = bounds[k + 3] - bounds[k];
        code |= spread10(quantise(centroid(r, k), bounds[k], ext)) << (2 - k);
    }
    keys[i] = code;
    vals[i] = i;
}

// Karras 2012: the common-prefix length of the keys (code, position); positions break ties, so all keys differ.
__device__ __forceinline__ int delta(const uint32_t* codes, int m, int i, int j) {
    if (j < 0 || j >= m) return -1;
    const uint32_t a = codes[i], b = codes[j];
    return a != b ? __clz(a ^ b) : 32 + __clz((uint32_t)(i ^ j));
}

// One thread per inner node i of m - 1 (m >= 2): its children, and their parents for the bottom-up pass.  Parents of
// inner nodes go to parent[0, m-1), of leaves to parent[m-1, 2m-1).
__global__ void __launch_bounds__(kTile) tlas_hierarchy_kernel(const uint32_t* __restrict__ codes, uint32_t m_, AccelNode* __restrict__ nodes,
                                                               int32_t* __restrict__ parent, uint32_t* __restrict__ arrivals) {
    const int m = (int)m_;
    const int i = blockIdx.x * kTile + threadIdx.x;
    if (m < 2 || i >= m - 1) return;
    const int d = delta(codes, m, i, i + 1) > delta(codes, m, i, i - 1) ? 1 : -1;
    const int dmin = delta(codes, m, i, i - d);
    int lmax = 2;
    while (delta(codes, m, i, i + lmax * d) > dmin) lmax <<= 1;
    int l = 0;
    for (int t = lmax >> 1; t >= 1; t >>= 1)
        if (delta(codes, m, i, i + (l + t) * d) > dmin) l += t;
    const int j = i + l * d;
    const int dnode = delta(codes, m, i, j);
    int s = 0;
    for (int div = 2;; div <<= 1) {
        const int t = (l + div - 1) / div;
        if (delta(codes, m, i, i + (s + t) * d) > dnode) s += t;
        if (t == 1) break;
    }
    const int split = i + s * d + (d < 0 ? -1 : 0);
    const int first = i < j ? i : j, last = i < j ? j : i;
    const int32_t c0 = first == split ? (int32_t)~(uint32_t)split : split;
    const int32_t c1 = last == split + 1 ? (int32_t)~(uint32_t)(split + 1) : split + 1;
    nodes[i].c0 = c0;
    nodes[i].c1 = c1;
    nodes[i].pad[0] = nodes[i].pad[1] = 0;
    parent[c0 < 0 ? (m - 1) + split : c0] = i;
    parent[c1 < 0 ? (m - 1) + split + 1 : c1] = i;
    arrivals[i] = 0;
}

// One thread per leaf (sorted position): its instance record in leaf order, then up the tree (arrive): the first arrival
// at a node stops, the second goes on with the node's box.
__global__ void __launch_bounds__(kTile) tlas_boxes_kernel(const AccelInstance* __restrict__ rec, const uint32_t* __restrict__ order, uint32_t m_,
                                                           AccelNode* nodes, AccelInstance* __restrict__ inst, const int32_t* __restrict__ parent,
                                                           uint32_t* arrivals) {
    const int m = (int)m_;
    const int i = blockIdx.x * kTile + threadIdx.x;
    if (m < 2) {  // the special roots of build_tree (k_accel.cu)
        if (i != 0) return;
        float lo[3], hi[3];
        empty_box(lo, hi);
        if (m == 1) {
            const AccelInstance r = rec[order[0]];
            inst[0] = r;
            for (int k = 0; k < 3; k++) {
                lo[k] = r.lo[k];
                hi[k] = r.hi[k];
            }
        }
        nodes[0] = special_root(lo, hi);
        return;
    }
    if (i >= m) return;
    const AccelInstance r = rec[order[i]];
    inst[i] = r;
    float lo[3] = {r.lo[0], r.lo[1], r.lo[2]}, hi[3] = {r.hi[0], r.hi[1], r.hi[2]};
    int32_t child = (int32_t)~(uint32_t)i;
    int node = parent[(m - 1) + i];
    while (true) {
        if (!arrive(nodes, arrivals, node, nodes[node].c0 == child ? 0 : 1, lo, hi)) return;
        if (node == 0) return;
        child = node;
        node = parent[node];
    }
}

}  // namespace

namespace tr {

void launch_block_scan(uint32_t* data, uint32_t len, cudaStream_t s) { tlas_scan_kernel<<<1, kScanThreads, 0, s>>>(data, len); }

// Host side: the top-level count, the instance checks and the buffer sizes come from what the host holds; nothing
// waits for the device unless a buffer grows.  The primitive table is on the device since tr_build_acceleration_structures
// (k_accel.cu accel_build), and a bottom-level refit keeps its boxes current (k_mesh_update.cu).
int32_t accel_build_tlas_async(tr_ctx* c) {
    if (!c->accel_blas_valid)
        return fail(TR_ERR_STATE, "top-level build: bottom-level structures missing (tr_build_acceleration_structures)");
    const uint32_t n = c->n_instances;
    uint32_t m = 0;
    for (uint32_t i = 0; i < n; i++) {  // the same checks, in the same order, as accel_build_tlas
        const uint32_t p = c->h_inst_prim[i];
        if (p >= c->n_primitives) return fail(TR_ERR_INVALID_ARG, "top-level build: instance %u refers to primitive %u of %u", i, p, c->n_primitives);
        if (c->h_prim_bucket[p] >= 2u || c->h_prim_tris[p] == 0u) continue;
        m++;
    }

    // scratch: records [m], keys [2][m], values [2][m], parents [2m], arrivals [m], digit counts [kRadix][tiles of m],
    // kept counts [tiles of n], centroid bounds [8]
    const uint32_t mc = m ? m : 1u, tiles_m = (mc + kTile - 1) / kTile, tiles_n = (n + kTile - 1) / kTile ? (n + kTile - 1) / kTile : 1u;
    ScratchLayout sl;
    const size_t off_rec = sl.take((size_t)mc * sizeof(AccelInstance)), off_keys = sl.take((size_t)mc * 8), off_vals = sl.take((size_t)mc * 8),
                 off_parent = sl.take((size_t)mc * 8), off_arr = sl.take((size_t)mc * 4), off_hist = sl.take((size_t)kRadix * tiles_m * 4),
                 off_cnt = sl.take((size_t)tiles_n * 4), off_bounds = sl.take(32);
    TR_TRY(c->accel_scratch.ensure(sl.bytes));
    TR_TRY(c->accel_tlas.ensure((size_t)(m >= 2 ? m - 1 : 1) * sizeof(AccelNode)));
    TR_TRY(c->accel_inst.ensure((size_t)mc * sizeof(AccelInstance)));
    char* base = c->accel_scratch.as<char>();
    AccelInstance* rec = reinterpret_cast<AccelInstance*>(base + off_rec);
    uint32_t* keys[2] = {reinterpret_cast<uint32_t*>(base + off_keys), reinterpret_cast<uint32_t*>(base + off_keys) + mc};
    uint32_t* vals[2] = {reinterpret_cast<uint32_t*>(base + off_vals), reinterpret_cast<uint32_t*>(base + off_vals) + mc};
    int32_t* parent = reinterpret_cast<int32_t*>(base + off_parent);
    uint32_t* arrivals = reinterpret_cast<uint32_t*>(base + off_arr);
    uint32_t* hist = reinterpret_cast<uint32_t*>(base + off_hist);
    uint32_t* cnt = reinterpret_cast<uint32_t*>(base + off_cnt);
    float* bounds = reinterpret_cast<float*>(base + off_bounds);
    const tr_instance* inst = c->instances.as<tr_instance>();
    const TlasPrim* prims = c->accel_prim_table.as<TlasPrim>();
    AccelNode* nodes = c->accel_tlas.as<AccelNode>();
    cudaStream_t s = c->stream;

    tlas_count_kernel<<<tiles_n, kTile, 0, s>>>(inst, n, prims, cnt);
    tlas_scan_kernel<<<1, kScanThreads, 0, s>>>(cnt, tiles_n);
    tlas_records_kernel<<<tiles_n, kTile, 0, s>>>(inst, n, prims, cnt, rec);
    tlas_bounds_kernel<<<1, kScanThreads, 0, s>>>(rec, m, bounds);
    tlas_codes_kernel<<<tiles_m, kTile, 0, s>>>(rec, m, bounds, keys[0], vals[0]);
    for (int pass = 0; pass < kRadixPasses; pass++) {  // an even number of passes: the sorted keys end in keys[0]
        const int in = pass & 1, shift = pass * kRadixBits;
        radix_histogram_kernel<<<tiles_m, kTile, 0, s>>>(keys[in], m, shift, hist);
        tlas_scan_kernel<<<1, kScanThreads, 0, s>>>(hist, kRadix * tiles_m);
        radix_scatter_kernel<<<tiles_m, kTile, 0, s>>>(keys[in], vals[in], m, shift, hist, keys[in ^ 1], vals[in ^ 1]);
    }
    tlas_hierarchy_kernel<<<tiles_m, kTile, 0, s>>>(keys[0], m, nodes, parent, arrivals);
    tlas_boxes_kernel<<<tiles_m, kTile, 0, s>>>(rec, vals[0], m, nodes, c->accel_inst.as<AccelInstance>(), parent, arrivals);
    count_launches(kAsyncTlasLaunches);
    TR_CUDA(cudaGetLastError());
    c->accel_n_instances = m;
    c->accel_tlas_valid = true;
    return TR_OK;
}

}  // namespace tr
