// k_accel_build.cu — the bottom-level acceleration structures built on the device, in stream order
// (tr_build_acceleration_structures_async).
//
// Reference behaviour: build_acceleration_structures_from_primitives (src/acceleration_structures.rs:6-104), one structure
// per primitive.  The host builder (k_accel.cu accel_build) reads the mesh back, waits, and runs a binned-SAH build; this
// one reads the positions and indices as the context's stream sees them and never waits.  The trees drop into the buffers
// the host build fills (the traversal of tr_device_accel.cuh, the refit of k_mesh_update.cu, both top-level builders):
//   - single-triangle leaves, so a primitive of nt >= 2 triangles has nt - 1 inner nodes, and the empty (nt = 0) and
//     one-leaf (nt = 1) roots of build_tree; every node range and triangle range is known on the host;
//   - each tree in preorder (root first, children after their parent), triangles in left-to-right leaf order;
//   - every inner box the exact union of its subtree (fminf / fmaxf), so every ray's bit is the definition's.
//
// Builder: H-PLOC (Benthin, Meister, Barczak, Mehalwal, Tsakok, Kensler, "H-PLOC: Hierarchical Parallel Locally-Ordered
// Clustering for Bounding Volume Hierarchy Construction", HPG 2024).  Every triangle gets a 30-bit Morton code normalised
// to its own primitive's centroid bounds; a stable LSD radix sort of (primitive, code) keeps each primitive's triangles
// together.  One thread per leaf climbs the implicit radix tree of the sorted keys (Apetrei 2014): the second thread to
// arrive at a node goes on.  A node whose range holds more than kPlocThreshold triangles, or a primitive's root, is
// reduced by its warp with PLOC (Meister & Bittner 2018) on the range's cluster list: nearest neighbour by the surface
// area of the union within kPlocRadius list positions, mutual pairs merge, until at most kPlocThreshold clusters remain
// (one at the root).  A range never crosses a primitive boundary.  Node ids come from an atomic counter; a final pass
// (one thread per node, walking up to its root) places every node at its preorder offset and every leaf at its
// triangle offset, so the output does not depend on which thread did what.
//
// Depth guard: H-PLOC's depth has no proven bound.  The placement pass records every primitive's depth; a primitive
// deeper than the limit (kAccelStack - 1, or TR_ACCEL_DEPTH_LIMIT) is built again, in the same launch sequence, as the
// plain radix tree over (code, position), whose depth is bounded (tr_device_accel.cuh).
//
// Launches (async_blas_launches): counts, 2 scans, init, bounds, codes, 5 per radix pass (histogram, chunk sums, chunk-sum scan, scan,
// scatter), then H-PLOC, placement, reset, H-PLOC, placement; the radix passes are ceil((30 + bits of the largest
// primitive id) / 8).
#include <algorithm>
#include <cstdlib>

#include "tr_device_build.cuh"
#include "tr_internal.h"

using namespace trd;

namespace {

constexpr int kScanChunk = kScanThreads * 4;   // entries per block of the two-level scan
constexpr int kPlocRadius = 8;
constexpr int kPlocThreshold = 16;     // two children's lists of at most 16 clusters fill a warp
constexpr uint32_t kInvalid = 0xffffffffu;
static_assert(2 * kPlocThreshold <= 32, "a node's two cluster lists fit in one warp");

struct BuildPrim {             // per primitive, assembled on the device (build_init_kernel)
    uint32_t first_index, nt;  // first index, triangles
    uint32_t tri_base;         // first leaf-order triangle = first sorted position
    uint32_t node_base;        // root node
    uint32_t keep;             // draw_buffer_index < 2 and nt != 0 (TlasPrim::keep)
    uint32_t pad[3];
};
static_assert(sizeof(BuildPrim) == 32, "BuildPrim");

// a cluster: its box and, in the spare words, the inner nodes and triangles below it
struct Cluster {
    float lo[3], hi[3];
    uint32_t inner, tris;
};

__device__ __forceinline__ void store_cluster(float4* cbox, uint32_t id, const Cluster& c) {
    cbox[2 * (size_t)id] = make_float4(c.lo[0], c.lo[1], c.lo[2], c.hi[0]);
    cbox[2 * (size_t)id + 1] = make_float4(c.hi[1], c.hi[2], __uint_as_float(c.inner), __uint_as_float(c.tris));
}

__device__ __forceinline__ Cluster load_cluster(const float4* cbox, uint32_t id) {   // L2: other blocks wrote it
    const float4 a = __ldcg(cbox + 2 * (size_t)id), b = __ldcg(cbox + 2 * (size_t)id + 1);
    Cluster c;
    c.lo[0] = a.x; c.lo[1] = a.y; c.lo[2] = a.z;
    c.hi[0] = a.w; c.hi[1] = b.x; c.hi[2] = b.y;
    c.inner = __float_as_uint(b.z);
    c.tris = __float_as_uint(b.w);
    return c;
}

// the primitive owning triangle g: the last whose tri_base <= g (primitives without triangles share their successor's)
__device__ __forceinline__ uint32_t prim_of(const BuildPrim* bp, uint32_t n_prims, uint32_t g) {
    return last_at_most(n_prims, g, [&](uint32_t p) { return __ldg(&bp[p].tri_base); });
}

__device__ __forceinline__ Cluster leaf_cluster(const Tri& t) {   // a leaf of one triangle
    Cluster c;
    empty_box(c.lo, c.hi);
    fold_tri(t, c.lo, c.hi);
    c.inner = 0;
    c.tris = 1;
    return c;
}

// float -> unsigned with the same order (NaN excluded by the callers; -0 maps to +0)
__device__ __forceinline__ uint32_t ordered(float x) {
    return x >= 0.0f ? __float_as_uint(__fadd_rn(x, 0.0f)) | 0x80000000u : ~__float_as_uint(x);
}
__device__ __forceinline__ float unordered(uint32_t u) { return __uint_as_float(u & 0x80000000u ? u & 0x7fffffffu : ~u); }

// scratch words
enum { W_COUNTER = 0, W_START = 1 };

// Launch 1: per primitive, its triangles and its node count; their exclusive scans (launches 2 and 3) are the first
// triangle and the root of every primitive, the offsets the host computes on its own for its checks and handles.
__global__ void __launch_bounds__(kTile) build_counts_kernel(const tr_primitive_info* __restrict__ prims, uint32_t n_prims,
                                                             uint32_t* __restrict__ tri_base, uint32_t* __restrict__ node_base) {
    const uint32_t p = blockIdx.x * kTile + threadIdx.x;
    if (p >= n_prims) return;
    const uint32_t nt = prims[p].index_count / 3u;
    tri_base[p] = nt;
    node_base[p] = nt > 1u ? nt - 1u : 1u;
}

// Launch 4: per primitive, its BuildPrim, the centroid bounds and depth start empty, and the nt <= 1 trees are written whole (build_tree:
// the empty root, or the leaf wrapped in a root whose second box is empty).  Per cluster id, no parent; per sorted
// position, the leaf is its own cluster list and no thread has reached its parent boundary yet.
__global__ void __launch_bounds__(kTile) build_init_kernel(const tr_primitive_info* __restrict__ prims, const uint32_t* __restrict__ tri_base,
                                                           const uint32_t* __restrict__ node_base, BuildPrim* __restrict__ bp,
                                                           uint32_t n_prims, uint32_t n,
                                                           const float* __restrict__ pos, const uint32_t* __restrict__ idx,
                                                           uint32_t* __restrict__ pbounds, uint32_t* __restrict__ pdepth,
                                                           uint32_t* __restrict__ words, int32_t* __restrict__ tparent,
                                                           uint32_t* __restrict__ cidx, int32_t* __restrict__ pidx,
                                                           AccelNode* __restrict__ nodes, float4* __restrict__ tris,
                                                           int32_t* __restrict__ parent, uint32_t* __restrict__ arrivals,
                                                           uint32_t* __restrict__ tri_src, TlasPrim* __restrict__ table) {
    const uint32_t i = blockIdx.x * kTile + threadIdx.x;
    if (i < 3 * n) tparent[i] = -1;
    if (i < n) {
        cidx[i] = i;
        pidx[i] = -1;
    }
    if (i == 0) words[W_COUNTER] = words[W_START] = 0u;
    if (i >= n_prims) return;
    for (int k = 0; k < 3; k++) {
        pbounds[i * 6 + k] = 0xffffffffu;
        pbounds[i * 6 + 3 + k] = 0u;
    }
    pdepth[i] = 0u;
    const tr_primitive_info pr = prims[i];
    BuildPrim b;
    b.first_index = pr.first_index;
    b.nt = pr.index_count / 3u;
    b.tri_base = tri_base[i];
    b.node_base = node_base[i];
    b.keep = pr.draw_buffer_index < 2u && b.nt != 0u;
    b.pad[0] = b.pad[1] = b.pad[2] = 0u;
    bp[i] = b;
    if (b.nt >= 2) return;
    float lo[3], hi[3];
    empty_box(lo, hi);
    if (b.nt == 1) {
        const Tri t = load_tri(pos, idx, b.first_index);
        fold_tri(t, lo, hi);
        for (int k = 0; k < 3; k++) tris[(size_t)b.tri_base * 3 + k] = t.v[k];
        tri_src[b.tri_base] = b.first_index;
    }
    nodes[b.node_base] = special_root(lo, hi);
    parent[b.node_base] = -1;
    arrivals[b.node_base] = 0u;
    table[i] = make_tlas_prim(lo, hi, b.node_base, b.tri_base, b.keep);
}

__device__ __forceinline__ void centroid(const Tri& t, float* c) {   // lo + hi, as build_range
    float tlo[3], thi[3];
    tri_box(t, tlo, thi);
    for (int k = 0; k < 3; k++) c[k] = tlo[k] + thi[k];
}

// Launch 2: every primitive's centroid bounds (NaN centroids left out)
__global__ void __launch_bounds__(kTile) build_bounds_kernel(const BuildPrim* __restrict__ bp, uint32_t n_prims, uint32_t n,
                                                             const float* __restrict__ pos, const uint32_t* __restrict__ idx,
                                                             uint32_t* __restrict__ pbounds) {
    const uint32_t g = blockIdx.x * kTile + threadIdx.x;
    if (g >= n) return;
    const uint32_t p = prim_of(bp, n_prims, g);
    const BuildPrim b = bp[p];
    float c[3];
    centroid(load_tri(pos, idx, b.first_index + (g - b.tri_base) * 3u), c);
    for (int k = 0; k < 3; k++) {
        if (!(c[k] == c[k])) continue;
        atomicMin(&pbounds[p * 6 + k], ordered(c[k]));
        atomicMax(&pbounds[p * 6 + 3 + k], ordered(c[k]));
    }
}

// Launch 3: keys (primitive << 30 | code) and values (triangle) in the initial order, which is (primitive, position)
__global__ void __launch_bounds__(kTile) build_codes_kernel(const BuildPrim* __restrict__ bp, uint32_t n_prims, uint32_t n,
                                                            const float* __restrict__ pos, const uint32_t* __restrict__ idx,
                                                            const uint32_t* __restrict__ pbounds, uint64_t* __restrict__ keys,
                                                            uint32_t* __restrict__ vals) {
    const uint32_t g = blockIdx.x * kTile + threadIdx.x;
    if (g >= n) return;
    const uint32_t p = prim_of(bp, n_prims, g);
    const BuildPrim b = bp[p];
    float c[3];
    centroid(load_tri(pos, idx, b.first_index + (g - b.tri_base) * 3u), c);
    uint32_t code = 0;
    for (int k = 0; k < 3; k++) {
        const uint32_t umn = pbounds[p * 6 + k], umx = pbounds[p * 6 + 3 + k];
        const float lo = umn == 0xffffffffu ? 0.0f : unordered(umn), hi = umx == 0u ? 0.0f : unordered(umx);
        code |= spread10(quantise(c[k], lo, hi - lo)) << (2 - k);
    }
    keys[g] = (uint64_t)p << 30 | code;
    vals[g] = g;
}

// The two-level scan of the radix sort's digit counts (tr_device_build.cuh): the sum of every chunk of kScanChunk
// entries, their one-block scan, then every chunk scanned from its offset.
__global__ void __launch_bounds__(kScanThreads) build_chunk_sums_kernel(const uint32_t* __restrict__ data, uint32_t len,
                                                                        uint32_t* __restrict__ sums) {
    __shared__ uint32_t warp_sum[32];
    const uint32_t base = blockIdx.x * kScanChunk + threadIdx.x * 4;
    uint32_t v = 0;
    for (int k = 0; k < 4; k++) v += base + k < len ? data[base + k] : 0u;
    uint32_t total;
    block_scan(v, warp_sum, &total);
    if (threadIdx.x == 0) sums[blockIdx.x] = total;
}

__global__ void __launch_bounds__(kScanThreads) build_scan_kernel(uint32_t* __restrict__ data, uint32_t len,
                                                                  const uint32_t* __restrict__ sums) {
    __shared__ uint32_t warp_sum[32];
    const uint32_t base = blockIdx.x * kScanChunk + threadIdx.x * 4;
    uint32_t v[4], t = 0;
    for (int k = 0; k < 4; k++) {
        v[k] = base + k < len ? data[base + k] : 0u;
        t += v[k];
    }
    uint32_t total;
    uint32_t x = sums[blockIdx.x] + block_scan(t, warp_sum, &total);
    for (int k = 0; k < 4; k++) {
        if (base + k < len) data[base + k] = x;
        x += v[k];
    }
}

// The boundary between sorted positions i and i + 1 of one primitive's segment [lo, hi]: the keys (code, position - lo)
// differ first at the highest bit of this xor.  Outside the segment: no boundary.
__device__ __forceinline__ uint64_t gap(const uint64_t* keys, uint32_t lo, uint32_t hi, uint32_t i) {
    if (i < lo || i >= hi) return ~0ull;
    const uint32_t a = (uint32_t)__ldg(keys + i) & 0x3fffffffu, b = (uint32_t)__ldg(keys + i + 1) & 0x3fffffffu;
    return (uint64_t)(a ^ b) << 32 | ((i - lo) ^ (i + 1 - lo));
}

__device__ __forceinline__ float union_area(const Cluster& a, const float* lo, const float* hi) {
    const float dx = fmaxf(a.hi[0], hi[0]) - fminf(a.lo[0], lo[0]);
    const float dy = fmaxf(a.hi[1], hi[1]) - fminf(a.lo[1], lo[1]);
    const float dz = fmaxf(a.hi[2], hi[2]) - fminf(a.lo[2], lo[2]);
    return __fadd_rn(__fadd_rn(__fmul_rn(dx, dy), __fmul_rn(dy, dz)), __fmul_rn(dz, dx));
}

struct Temp {       // what a merge writes per new node: its children (cluster ids), what lies below its first child
    int32_t c0, c1;
    uint32_t inner0, tris0;
};

// The thread that owns a node reduces the cluster lists of its two children (ranges [l, split] and [split + 1, r]) with
// PLOC until at most `target` clusters remain, and stores the list at l.  A list is compacted at the start of its range and
// ends at the first kInvalid, or after min(size, threshold) entries; two lists hold at most 2 kPlocThreshold clusters.
// Pair keys (area, lower position, higher position) order all pairs, so the smallest pair in reach is mutual and every
// round merges at least one.
__device__ __forceinline__ void ploc_merge(uint32_t l, uint32_t r, uint32_t split, uint32_t threshold, uint32_t target, uint32_t n_leaves,
                           uint32_t prim, uint32_t* cidx, float4* cbox, int32_t* tparent, Temp* tnode, uint32_t* tprim,
                           uint32_t* counter) {
    constexpr int kMax = 2 * kPlocThreshold;
    uint32_t ids[kMax];
    Cluster cl[kMax];
    uint32_t n = 0;
    for (uint32_t j = 0; j < min(split - l + 1, threshold); j++) {
        const uint32_t v = __ldcg(cidx + l + j);
        if (v == kInvalid) break;
        ids[n++] = v;
    }
    for (uint32_t j = 0; j < min(r - split, threshold); j++) {
        const uint32_t v = __ldcg(cidx + split + 1 + j);
        if (v == kInvalid) break;
        ids[n++] = v;
    }
    for (uint32_t j = 0; j < n; j++) cl[j] = load_cluster(cbox, ids[j]);
    while (n > target) {
        uint8_t nn[kMax];
        uint32_t makers = 0;
#pragma unroll 1   // rolled: unrolled, the candidate loops spill
        for (uint32_t a = 0; a < n; a++) {
            uint64_t best = ~0ull;
            const uint32_t b0 = a > (uint32_t)kPlocRadius ? a - kPlocRadius : 0u, b1 = min(n, a + kPlocRadius + 1);
#pragma unroll 1
            for (uint32_t b = b0; b < b1; b++) {
                if (b == a) continue;
                const float area = union_area(cl[a], cl[b].lo, cl[b].hi);
                const uint32_t bits = area >= 0.0f ? __float_as_uint(__fadd_rn(area, 0.0f)) : 0x7fffffffu;   // NaN last
                const uint64_t key = (uint64_t)bits << 10 | min(a, b) << 5 | max(a, b);
                if (key < best) best = key;
            }
            const uint32_t lo = (uint32_t)(best >> 5) & 31, hi = (uint32_t)best & 31;
            nn[a] = (uint8_t)(lo == a ? hi : lo);
        }
        for (uint32_t a = 0; a < n; a++) makers += nn[nn[a]] == a && a < nn[a];
        uint32_t t = atomicAdd(counter, makers), w = 0;
        for (uint32_t a = 0; a < n; a++) {   // in place: w <= a, and a merge partner lies above a
            const uint32_t b = nn[a];
            const bool mutual = nn[b] == a;
            if (mutual && a > b) continue;
            if (mutual) {
                tnode[t] = Temp{(int32_t)ids[a], (int32_t)ids[b], cl[a].inner, cl[a].tris};
                tprim[t] = prim;
                tparent[ids[a]] = (int32_t)t;
                tparent[ids[b]] = (int32_t)t;
                Cluster m;
                for (int k = 0; k < 3; k++) {
                    m.lo[k] = fminf(cl[a].lo[k], cl[b].lo[k]);
                    m.hi[k] = fmaxf(cl[a].hi[k], cl[b].hi[k]);
                }
                m.inner = cl[a].inner + cl[b].inner + 1u;
                m.tris = cl[a].tris + cl[b].tris;
                ids[w] = n_leaves + t;
                cl[w] = m;
                store_cluster(cbox, n_leaves + t, m);
                t++;
            } else {
                ids[w] = ids[a];
                cl[w] = cl[a];
            }
            w++;
        }
        n = w;
    }
    for (uint32_t j = 0; j < min(r - l + 1, (uint32_t)kMax); j++) cidx[l + j] = j < n ? ids[j] : kInvalid;
}

// One thread per sorted position of the primitives being built (pass 0: every primitive of >= 2 triangles; pass 1: those
// deeper than `depth_limit`, with threshold 1, i.e. the radix tree).  Apetrei's climb: at a boundary the left child leaves
// its l, the right child its r; the second to arrive takes the other's and owns the parent.
__global__ void __launch_bounds__(kTile) build_hploc_kernel(const uint64_t* __restrict__ keys, const uint32_t* __restrict__ vals,
                                                            uint32_t n, const BuildPrim* __restrict__ bp, const float* __restrict__ pos,
                                                            const uint32_t* __restrict__ idx, const uint32_t* __restrict__ pdepth,
                                                            uint32_t depth_limit, int pass, int32_t* pidx, uint32_t* cidx,
                                                            float4* cbox, int32_t* __restrict__ tparent, Temp* __restrict__ tnode,
                                                            uint32_t* __restrict__ tprim, uint32_t* counter) {
    const uint32_t s = blockIdx.x * kTile + threadIdx.x;
    if (s >= n) return;
    const uint32_t p = (uint32_t)(__ldg(keys + s) >> 30);
    const BuildPrim b = bp[p];
    if (b.nt < 2 || (pass != 0 && pdepth[p] <= depth_limit)) return;
    const uint32_t lo = b.tri_base, hi = b.tri_base + b.nt - 1;
    store_cluster(cbox, s, leaf_cluster(load_tri(pos, idx, b.first_index + (__ldg(vals + s) - b.tri_base) * 3u)));
    const uint32_t threshold = pass == 0 ? kPlocThreshold : 1u;
    uint32_t l = s, r = s;
    while (true) {
        __threadfence();   // this range's cluster list and boxes before the exchange that hands them on
        const uint64_t gl = l > lo ? gap(keys, lo, hi, l - 1) : ~0ull, gr = gap(keys, lo, hi, r);
        uint32_t split;
        int32_t prev;
        if (gr < gl) {   // the parent extends to the right: this node is its left child
            split = r;
            prev = atomicExch(&pidx[split], (int32_t)l);
            if (prev >= 0) r = (uint32_t)prev;
        } else {
            split = l - 1;
            prev = atomicExch(&pidx[split], (int32_t)r);
            if (prev >= 0) l = (uint32_t)prev;
        }
        if (prev < 0) return;   // the sibling is not done yet: it goes on from here
        __threadfence();
        const bool root = l == lo && r == hi;
        if (r - l + 1 > threshold || root)
            ploc_merge(l, r, split, threshold, root ? 1u : threshold, n, p, cidx, cbox, tparent, tnode, tprim, counter);
        if (root) return;
    }
}

// Placement, one thread per node made in this pass (ids [start, counter)): up to the root, summing the preorder offset
// (1 for the parent, plus the inner nodes of the left sibling for a right child) and the triangle offset (the left
// sibling's triangles).  It writes the node, the triangles of its leaf children, the refit tables and, at a root, the
// primitive's TlasPrim.  Pass 0 records every primitive's depth (inner nodes on the longest path).
__global__ void __launch_bounds__(kTile) build_place_kernel(uint32_t n, const uint32_t* __restrict__ words, const Temp* __restrict__ tnode,
                                                            const int32_t* __restrict__ tparent, const uint32_t* __restrict__ tprim,
                                                            const float4* __restrict__ cbox, const BuildPrim* __restrict__ bp,
                                                            const uint32_t* __restrict__ vals, const float* __restrict__ pos,
                                                            const uint32_t* __restrict__ idx, int pass, uint32_t* __restrict__ pdepth,
                                                            AccelNode* __restrict__ nodes, float4* __restrict__ tris,
                                                            int32_t* __restrict__ parent, uint32_t* __restrict__ arrivals,
                                                            uint32_t* __restrict__ tri_src, TlasPrim* __restrict__ table) {
    const uint32_t t = words[W_START] + blockIdx.x * kTile + threadIdx.x;
    if (t >= words[W_COUNTER]) return;
    uint32_t pre = 0, toff = 0, depth = 1;
    uint32_t x = n + t;
    for (int32_t up = tparent[x]; up >= 0; up = tparent[x]) {
        const Temp u = tnode[up];
        pre += 1u;
        if ((uint32_t)u.c1 == x) {
            pre += u.inner0;
            toff += u.tris0;
        }
        depth++;
        x = n + (uint32_t)up;
    }
    const uint32_t prim = tprim[t];
    const BuildPrim b = bp[prim];
    const uint32_t self = b.node_base + pre;
    const Temp me = tnode[t];
    const Cluster k0 = load_cluster(cbox, (uint32_t)me.c0), k1 = load_cluster(cbox, (uint32_t)me.c1);
    AccelNode out;
    for (int k = 0; k < 3; k++) {
        out.lo0[k] = k0.lo[k]; out.hi0[k] = k0.hi[k];
        out.lo1[k] = k1.lo[k]; out.hi1[k] = k1.hi[k];
    }
    out.pad[0] = out.pad[1] = 0u;
    const uint32_t child[2] = {(uint32_t)me.c0, (uint32_t)me.c1};
    const uint32_t child_pre[2] = {self + 1u, self + 1u + me.inner0};
    const uint32_t child_tri[2] = {toff, toff + me.tris0};
    int32_t ref[2];
    for (int side = 0; side < 2; side++) {
        if (child[side] >= n) {
            ref[side] = (int32_t)child_pre[side];
            parent[child_pre[side]] = (int32_t)self;
        } else {   // a leaf: one triangle, at child_tri of the primitive's leaf order
            const uint32_t lt = child_tri[side], first = b.first_index + (vals[child[side]] - b.tri_base) * 3u;
            ref[side] = (int32_t)~lt;
            const Tri tr = load_tri(pos, idx, first);
            for (int k = 0; k < 3; k++) tris[(size_t)(b.tri_base + lt) * 3 + k] = tr.v[k];
            tri_src[b.tri_base + lt] = first;
        }
    }
    out.c0 = ref[0];
    out.c1 = ref[1];
    nodes[self] = out;
    arrivals[self] = 0u;
    if (pre == 0) {   // the root
        parent[self] = -1;
        float lo[3], hi[3];
        for (int k = 0; k < 3; k++) {
            lo[k] = fminf(k0.lo[k], k1.lo[k]);
            hi[k] = fmaxf(k0.hi[k], k1.hi[k]);
        }
        table[prim] = make_tlas_prim(lo, hi, b.node_base, b.tri_base, b.keep);
    }
    if (pass == 0) atomicMax(&pdepth[prim], depth);
}

// Between the passes: the positions of every primitive deeper than the limit start over, and pass 1's ids follow pass 0's
__global__ void __launch_bounds__(kTile) build_reset_kernel(const uint64_t* __restrict__ keys, uint32_t n, const uint32_t* __restrict__ pdepth,
                                                            uint32_t depth_limit, uint32_t* __restrict__ words, uint32_t* __restrict__ cidx,
                                                            int32_t* __restrict__ pidx) {
    const uint32_t s = blockIdx.x * kTile + threadIdx.x;
    if (s == 0) words[W_START] = words[W_COUNTER];
    if (s >= n || pdepth[(uint32_t)(keys[s] >> 30)] <= depth_limit) return;
    cidx[s] = s;
    pidx[s] = -1;
}

uint32_t radix_passes(uint32_t n_prims) {
    uint32_t bits = 0;
    while (bits < 32 && (n_prims - 1u) >> bits) bits++;
    return (30u + bits + kRadixBits - 1) / kRadixBits;
}

}  // namespace

namespace tr {

int async_blas_launches(uint32_t n_primitives) { return 11 + 5 * (int)radix_passes(n_primitives); }

// Host side: every count, offset and error comes from what the host holds (tr_set_mesh checked the indices against the
// vertices; tr_set_primitives keeps the index ranges and draw buffers); nothing waits for the device unless a buffer grows.
int32_t accel_build_async(tr_ctx* c) {
    static const char* who = "tr_build_acceleration_structures_async";
    if (!c->n_vertices || !c->n_indices) return fail(TR_ERR_STATE, "%s: mesh not set", who);
    if (!c->n_primitives) return fail(TR_ERR_STATE, "%s: primitives not set", who);
    const uint32_t np = c->n_primitives;
    std::vector<uint32_t> root(np), tri_base(np);
    uint64_t n = 0, nn = 0;
    for (uint32_t p = 0; p < np; p++) {   // the checks of accel_build, in its order
        const uint32_t nt = c->h_prim_count[p] / 3;
        if ((uint64_t)c->h_prim_first[p] + c->h_prim_count[p] > c->n_indices)
            return fail(TR_ERR_INVALID_ARG, "tr_build_acceleration_structures: primitive %u indexes past the index buffer", p);
        if (nt >= (1u << 28)) return fail(TR_ERR_UNSUPPORTED, "tr_build_acceleration_structures: primitive %u has %u triangles", p, nt);
        tri_base[p] = (uint32_t)n;
        root[p] = (uint32_t)nn;
        n += nt;
        nn += nt > 1 ? nt - 1 : 1;
    }
    if (n >= (1u << 29)) return fail(TR_ERR_UNSUPPORTED, "%s: %llu triangles (at most 2^29 - 1)", who, (unsigned long long)n);
    const uint32_t nc = n ? (uint32_t)n : 1u, tiles = (nc + kTile - 1) / kTile, hist_len = kRadix * tiles,
                   chunks = (hist_len + kScanChunk - 1) / kScanChunk;

    // scratch: primitives [np], centroid bounds [6 np], depths [np], words [4], keys [2][n] (8 B), values [2][n], digit
    // counts [hist_len], chunk sums [chunks], cluster lists [n], boundary slots [n], cluster boxes [3n] (32 B), parents of
    // clusters [3n], nodes made [2n] (16 B), their primitives [2n]
    ScratchLayout sl;
    const size_t o_bp = sl.take((size_t)np * sizeof(BuildPrim)), o_counts = sl.take((size_t)np * 8), o_bounds = sl.take((size_t)np * 24),
                 o_depth = sl.take((size_t)np * 4), o_words = sl.take(16), o_keys = sl.take((size_t)nc * 16), o_vals = sl.take((size_t)nc * 8),
                 o_hist = sl.take((size_t)hist_len * 4), o_sums = sl.take((size_t)chunks * 4), o_cidx = sl.take((size_t)nc * 4),
                 o_pidx = sl.take((size_t)nc * 4), o_cbox = sl.take((size_t)nc * 96), o_tparent = sl.take((size_t)nc * 12),
                 o_tnode = sl.take((size_t)nc * 2 * sizeof(Temp)), o_tprim = sl.take((size_t)nc * 8);
    TR_TRY(c->accel_build_scratch.ensure(sl.bytes));
    TR_TRY(c->accel_blas.ensure((size_t)nn * sizeof(AccelNode)));
    TR_TRY(c->accel_tris.ensure((size_t)nc * 3 * sizeof(float4)));
    TR_TRY(c->accel_prim_table.ensure((size_t)np * sizeof(TlasPrim)));
    TR_TRY(c->accel_refit.ensure((size_t)(nn * 2 + n) * 4));
    char* base = c->accel_build_scratch.as<char>();
    BuildPrim* d_bp = reinterpret_cast<BuildPrim*>(base + o_bp);
    uint32_t* d_tri_base = reinterpret_cast<uint32_t*>(base + o_counts);
    uint32_t* d_node_base = d_tri_base + np;
    const tr_primitive_info* prims = c->primitives.as<tr_primitive_info>();
    uint32_t* bounds = reinterpret_cast<uint32_t*>(base + o_bounds);
    uint32_t* depth = reinterpret_cast<uint32_t*>(base + o_depth);
    uint32_t* d_words = reinterpret_cast<uint32_t*>(base + o_words);
    uint64_t* keys[2] = {reinterpret_cast<uint64_t*>(base + o_keys), reinterpret_cast<uint64_t*>(base + o_keys) + nc};
    uint32_t* vals[2] = {reinterpret_cast<uint32_t*>(base + o_vals), reinterpret_cast<uint32_t*>(base + o_vals) + nc};
    uint32_t* hist = reinterpret_cast<uint32_t*>(base + o_hist);
    uint32_t* sums = reinterpret_cast<uint32_t*>(base + o_sums);
    uint32_t* cidx = reinterpret_cast<uint32_t*>(base + o_cidx);
    int32_t* pidx = reinterpret_cast<int32_t*>(base + o_pidx);
    float4* cbox = reinterpret_cast<float4*>(base + o_cbox);
    int32_t* tparent = reinterpret_cast<int32_t*>(base + o_tparent);
    Temp* tnode = reinterpret_cast<Temp*>(base + o_tnode);
    uint32_t* tprim = reinterpret_cast<uint32_t*>(base + o_tprim);
    AccelNode* nodes = c->accel_blas.as<AccelNode>();
    float4* tris = c->accel_tris.as<float4>();
    int32_t* parent = c->accel_refit.as<int32_t>();
    uint32_t* arrivals = c->accel_refit.as<uint32_t>() + nn;
    uint32_t* tri_src = arrivals + nn;
    TlasPrim* table = c->accel_prim_table.as<TlasPrim>();
    const float* pos = c->mesh_pos.as<float>();
    const uint32_t* idx = c->mesh_idx.as<uint32_t>();
    const char* env = getenv("TR_ACCEL_DEPTH_LIMIT");
    const uint32_t depth_limit = env ? (uint32_t)strtoul(env, nullptr, 10) : (uint32_t)(kAccelStack - 1);
    const uint32_t nu = (uint32_t)n, init_items = std::max(3 * nc, np);
    cudaStream_t s = c->stream;

    build_counts_kernel<<<(np + kTile - 1) / kTile, kTile, 0, s>>>(prims, np, d_tri_base, d_node_base);
    launch_block_scan(d_tri_base, np, s);
    launch_block_scan(d_node_base, np, s);
    build_init_kernel<<<(init_items + kTile - 1) / kTile, kTile, 0, s>>>(prims, d_tri_base, d_node_base, d_bp, np, nu, pos, idx, bounds, depth, d_words, tparent,
                                                                         cidx, pidx, nodes, tris, parent, arrivals, tri_src, table);
    build_bounds_kernel<<<tiles, kTile, 0, s>>>(d_bp, np, nu, pos, idx, bounds);
    build_codes_kernel<<<tiles, kTile, 0, s>>>(d_bp, np, nu, pos, idx, bounds, keys[0], vals[0]);
    const int passes = (int)radix_passes(np);
    for (int pass = 0; pass < passes; pass++) {
        const int in = pass & 1, shift = pass * kRadixBits;
        radix_histogram_kernel<<<tiles, kTile, 0, s>>>(keys[in], nu, shift, hist);
        build_chunk_sums_kernel<<<chunks, kScanThreads, 0, s>>>(hist, hist_len, sums);
        launch_block_scan(sums, chunks, s);
        build_scan_kernel<<<chunks, kScanThreads, 0, s>>>(hist, hist_len, sums);
        radix_scatter_kernel<<<tiles, kTile, 0, s>>>(keys[in], vals[in], nu, shift, hist, keys[in ^ 1], vals[in ^ 1]);
    }
    const int out = passes & 1;
    for (int pass = 0; pass < 2; pass++) {
        if (pass == 1) build_reset_kernel<<<tiles, kTile, 0, s>>>(keys[out], nu, depth, depth_limit, d_words, cidx, pidx);
        build_hploc_kernel<<<tiles, kTile, 0, s>>>(keys[out], vals[out], nu, d_bp, pos, idx, depth, depth_limit, pass, pidx, cidx,
                                                      cbox, tparent, tnode, tprim, d_words + W_COUNTER);
        build_place_kernel<<<tiles, kTile, 0, s>>>(nu, d_words, tnode, tparent, tprim, cbox, d_bp, vals[out], pos, idx, pass, depth,
                                                      nodes, tris, parent, arrivals, tri_src, table);
    }
    count_launches(async_blas_launches(np));
    TR_CUDA(cudaGetLastError());

    c->h_prim_root.resize(np);
    c->h_prim_tri_base.resize(np);
    for (uint32_t p = 0; p < np; p++) {
        c->h_prim_root[p] = root[p];
        c->h_prim_tri_base[p] = tri_base[p];
    }
    c->accel_blas_nodes = (uint32_t)nn;
    c->accel_n_tris = nu;
    c->accel_blas_valid = true;
    return accel_build_tlas_async(c);
}

}  // namespace tr
