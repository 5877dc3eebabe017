// k_mesh_update.cu — what depends on the vertex positions besides the rasteriser's own reads, recomputed on the device in
// stream order: the culling spheres of the binning pass (ensure_chunks, tr_update_mesh_vertices) and the bottom-level
// acceleration structures (tr_update_mesh_vertices after tr_build_acceleration_structures).
//
// Chunk spheres: one per TR_CHUNK_TRIS consecutive triangles of every primitive, the box of the chunk's vertices in double,
// centre 0.5 (lo + hi), radius to the farthest vertex in double, widened by the centre's rounding to float and by 1 + 1e-6.
// The results are bytes that tests restate in numpy, so every operation is an unfused IEEE one (__dadd_rn, __dmul_rn) in
// the order of the formula, and the box folds keep the first of two equal extremes (-0 against +0), as a sequential
// `lo = min(lo, v)` over the chunk's indices does.
//
// Refit: the mesh keeps its topology, so every tree of tr_build_acceleration_structures keeps its nodes and leaf ranges; only
// the triangles (gathered again from the positions in leaf order) and the boxes change.  The boxes are recomputed
// bottom-up with per-node arrival counters (arrive, tr_device_build.cuh); fminf / fmaxf are exact, so every inner box is
// the exact union of its subtree (the sign of a zero may depend on the arrival order; the slab test cannot see it).  The
// depth is the build's, below kAccelStack.  Two launches whatever the mesh size: gather, boxes.
#include "tr_device_build.cuh"
#include "tr_internal.h"

using namespace trd;

namespace {

constexpr int kChunkWarps = 4;       // chunks per block of the sphere kernel (one warp each)
constexpr int kRefitThreads = 256;

// first of two equal values wins: the order-preserving folds of a sequential std::min / std::max
__device__ __forceinline__ double min_first(double a, double b) { return b < a ? b : a; }
__device__ __forceinline__ double max_first(double a, double b) { return a < b ? b : a; }

// One warp per chunk.  Lane l takes the chunk's triangles 2l and 2l + 1 (indices [6l, 6l + 6) of the chunk), folds them in
// order, and the lanes combine with shuffles at offsets 1, 2, 4, 8, 16: lane 0 then holds the fold of lanes 0..31 in
// lane order, i.e. the sequential fold over the chunk.  The radius is a maximum of non-negative values, in any order.
__global__ void __launch_bounds__(kChunkWarps * 32) chunk_spheres_kernel(const float* __restrict__ pos, const uint32_t* __restrict__ idx,
                                                                         const tr_primitive_info* __restrict__ prims,
                                                                         const uint32_t* __restrict__ base, uint32_t n_prims,
                                                                         uint32_t n_chunks, float4* __restrict__ out) {
    const uint32_t chunk = blockIdx.x * kChunkWarps + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (chunk >= n_chunks) return;
    const uint32_t p = last_at_most(n_prims, chunk, [&](uint32_t q) { return __ldg(base + q); });   // the chunk's primitive
    const tr_primitive_info pr = prims[p];
    const uint32_t tris = pr.index_count / 3u, t0 = (chunk - __ldg(base + p)) * TR_CHUNK_TRIS;
    const uint32_t t1 = min(t0 + TR_CHUNK_TRIS, tris);
    const uint32_t i0 = pr.first_index + t0 * 3u, i1 = pr.first_index + t1 * 3u;
    const uint32_t my0 = min(i0 + lane * 6u, i1), my1 = min(my0 + 6u, i1);

    float v[6][3];
    double lo[3] = {1e300, 1e300, 1e300}, hi[3] = {-1e300, -1e300, -1e300};
#pragma unroll
    for (int j = 0; j < 6; j++) {
        if (my0 + j < my1) {
            const uint32_t vi = __ldg(idx + my0 + j);
            v[j][0] = __ldg(pos + (size_t)vi * 3);
            v[j][1] = __ldg(pos + (size_t)vi * 3 + 1);
            v[j][2] = __ldg(pos + (size_t)vi * 3 + 2);
#pragma unroll
            for (int k = 0; k < 3; k++) {
                lo[k] = min_first(lo[k], (double)v[j][k]);
                hi[k] = max_first(hi[k], (double)v[j][k]);
            }
        }
    }
#pragma unroll
    for (int o = 1; o < 32; o <<= 1)
#pragma unroll
        for (int k = 0; k < 3; k++) {   // lane + o >= 32 reads its own value: a no-op fold
            lo[k] = min_first(lo[k], __shfl_down_sync(0xffffffffu, lo[k], o));
            hi[k] = max_first(hi[k], __shfl_down_sync(0xffffffffu, hi[k], o));
        }
    double cen[3];
#pragma unroll
    for (int k = 0; k < 3; k++) {
        lo[k] = __shfl_sync(0xffffffffu, lo[k], 0);
        hi[k] = __shfl_sync(0xffffffffu, hi[k], 0);
        cen[k] = __dmul_rn(0.5, __dadd_rn(lo[k], hi[k]));
    }
    double r2 = 0.0;
#pragma unroll
    for (int j = 0; j < 6; j++) {
        if (my0 + j < my1) {
            const double dx = __dsub_rn((double)v[j][0], cen[0]), dy = __dsub_rn((double)v[j][1], cen[1]),
                         dz = __dsub_rn((double)v[j][2], cen[2]);
            r2 = max_first(r2, __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz)));
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) r2 = max_first(r2, __shfl_xor_sync(0xffffffffu, r2, o));
    if (lane != 0) return;
    const float fc[3] = {__double2float_rn(cen[0]), __double2float_rn(cen[1]), __double2float_rn(cen[2])};
    // the centre was rounded to float: widen the radius by that much and by its own rounding
    const double shift = __dadd_rn(__dadd_rn(fabs(__dsub_rn((double)fc[0], cen[0])), fabs(__dsub_rn((double)fc[1], cen[1]))),
                                   fabs(__dsub_rn((double)fc[2], cen[2])));
    float r = __double2float_rn(__dmul_rn(__dadd_rn(__dsqrt_rn(r2), shift), 1.0 + 1e-6));
    if (!(r == r) || isinf(r)) r = __int_as_float(0x7f800000);   // non-finite vertices: never culled
    out[chunk] = make_float4(fc[0], fc[1], fc[2], r);
}

// Refit, launch 1: every leaf-order triangle again from the positions (the layout of accel_build), and the arrival
// counters of the boxes pass back to zero.
__global__ void __launch_bounds__(kRefitThreads) blas_gather_kernel(const float* __restrict__ pos, const uint32_t* __restrict__ idx,
                                                                    const uint32_t* __restrict__ tri_src, uint32_t n_tris,
                                                                    float4* __restrict__ tris, uint32_t* __restrict__ arrivals,
                                                                    uint32_t n_nodes) {
    const uint32_t i = blockIdx.x * kRefitThreads + threadIdx.x;
    if (i < n_nodes) arrivals[i] = 0u;
    if (i >= n_tris) return;
    const Tri t = load_tri(pos, idx, tri_src[i]);
    for (int k = 0; k < 3; k++) tris[(size_t)i * 3 + k] = t.v[k];
}

// the box of a leaf's triangles (up to 4: the refit also runs on trees of the host builder)
__device__ __forceinline__ void leaf_box(const float4* __restrict__ tris, uint32_t tri_base, int32_t ref, float* lo, float* hi) {
    const uint32_t code = ~(uint32_t)ref, first = code & 0x0fffffffu, count = (code >> 28) + 1u;
    empty_box(lo, hi);
    for (uint32_t j = 0; j < count; j++) {
        const float4* t = tris + (size_t)(tri_base + first + j) * 3;
        fold_tri(Tri{{t[0], t[1], t[2]}}, lo, hi);
    }
}

// Refit, launch 2: one thread per node.  It stores the boxes of its leaf children.  A node whose two children are leaves
// is complete at once; with one leaf child the thread arrives at its own node like a child would.  A thread that completes
// a node goes on upwards: it stores the node's box in its parent and arrives there; the first arrival stops, the second
// unions both boxes and goes on.  At a root it writes the primitive's box into the top level's primitive table.
__global__ void __launch_bounds__(kRefitThreads) blas_boxes_kernel(AccelNode* nodes, const int32_t* __restrict__ parent, uint32_t* arrivals,
                                                                   uint32_t n_nodes, const float4* __restrict__ tris,
                                                                   const tr_primitive_info* __restrict__ prims, TlasPrim* table,
                                                                   uint32_t n_prims) {
    const uint32_t i = blockIdx.x * kRefitThreads + threadIdx.x;
    if (i >= n_nodes) return;
    // the node's primitive: the last whose root is <= i (the trees lie in primitive order)
    const uint32_t p = last_at_most(n_prims, i, [&](uint32_t q) { return table[q].blas_root; });
    const uint32_t tri_base = table[p].tri_base;
    AccelNode* n = nodes + i;
    const int32_t c0 = n->c0, c1 = n->c1;
    float lo[3], hi[3];
    if (c0 == c1) {   // the special roots of build_tree (k_accel.cu): the empty tree, or one leaf wrapped in a root
        if (prims[p].index_count / 3u == 0u) return;   // empty: both boxes stay empty, and so does the primitive's box
        leaf_box(tris, tri_base, c0, lo, hi);
        store_box(n, 0, lo, hi);                        // the second box stays empty
    } else if (c0 < 0 && c1 < 0) {   // two leaf children: the node is complete
        float lo1[3], hi1[3];
        leaf_box(tris, tri_base, c0, lo, hi);
        store_box(n, 0, lo, hi);
        leaf_box(tris, tri_base, c1, lo1, hi1);
        store_box(n, 1, lo1, hi1);
        for (int k = 0; k < 3; k++) {
            lo[k] = fminf(lo[k], lo1[k]);
            hi[k] = fmaxf(hi[k], hi1[k]);
        }
    } else if (c0 < 0 || c1 < 0) {   // one leaf child: its box arrives at this node as the inner child's will
        const int side = c0 < 0 ? 0 : 1;
        leaf_box(tris, tri_base, side ? c1 : c0, lo, hi);
        if (!arrive(nodes, arrivals, (int)i, side, lo, hi)) return;
    } else {
        return;   // both children inner: their threads arrive here
    }
    int32_t node = (int32_t)i;
    while (true) {   // `node` is complete and (lo, hi) is its box
        const int32_t up = parent[node];
        if (up < 0) {
            TlasPrim* t = table + p;
            for (int k = 0; k < 3; k++) {
                t->lo[k] = lo[k];
                t->hi[k] = hi[k];
            }
            return;
        }
        if (!arrive(nodes, arrivals, up, nodes[up].c0 == node ? 0 : 1, lo, hi)) return;
        node = up;
    }
}

}  // namespace

namespace tr {

int32_t launch_chunk_spheres(tr_ctx* c) {
    if (!c->n_chunks) return TR_OK;
    chunk_spheres_kernel<<<(c->n_chunks + kChunkWarps - 1) / kChunkWarps, kChunkWarps * 32, 0, c->stream>>>(
        c->mesh_pos.as<float>(), c->mesh_idx.as<uint32_t>(), c->primitives.as<tr_primitive_info>(), c->prim_chunk_base.as<uint32_t>(),
        c->n_primitives, c->n_chunks, c->chunk_spheres.as<float4>());
    count_launches(kChunkSphereLaunches);
    TR_CUDA(cudaGetLastError());
    return TR_OK;
}

int32_t accel_refit_blas(tr_ctx* c) {
    const uint32_t nn = c->accel_blas_nodes, nt = c->accel_n_tris, grid = nn > nt ? nn : nt;
    uint32_t* parent = c->accel_refit.as<uint32_t>();
    uint32_t* arrivals = parent + nn;
    const uint32_t* tri_src = arrivals + nn;
    blas_gather_kernel<<<(grid + kRefitThreads - 1) / kRefitThreads, kRefitThreads, 0, c->stream>>>(
        c->mesh_pos.as<float>(), c->mesh_idx.as<uint32_t>(), tri_src, nt, c->accel_tris.as<float4>(), arrivals, nn);
    blas_boxes_kernel<<<(nn + kRefitThreads - 1) / kRefitThreads, kRefitThreads, 0, c->stream>>>(
        c->accel_blas.as<AccelNode>(), reinterpret_cast<const int32_t*>(parent), arrivals, nn, c->accel_tris.as<float4>(),
        c->primitives.as<tr_primitive_info>(), c->accel_prim_table.as<TlasPrim>(), c->n_primitives);
    count_launches(kRefitLaunches);
    TR_CUDA(cudaGetLastError());
    return TR_OK;
}

}  // namespace tr
