// tr_device_build.cuh — building blocks of the device-side tree writers: the top-level build (k_accel_device.cu), the
// bottom-level build (k_accel_build.cu) and the bottom-level refit (k_mesh_update.cu).
//
// Every piece here is exactness-critical.  The box folds are the host builder's (k_accel.cu box_grow / box_union) byte for
// byte; the arrival step's fences and their order keep a box from being read before it is written; the radix scatter is
// stable, which the builders' tie-breaking, and with it their depth bounds (tr_device_accel.cuh), rely on.
#pragma once

#include "tr_device_accel.cuh"

namespace trd {

constexpr int kTile = 256;          // items per block of the per-item kernels, and per tile of the radix sort
constexpr int kRadixBits = 8;
constexpr int kRadix = 1 << kRadixBits;
constexpr int kScanThreads = 1024;  // threads of a block-wide scan
static_assert(kTile == kRadix, "the histogram kernel keeps one digit per thread");

// Morton codes: 10 bits -> every third bit of 30
TRD uint32_t spread10(uint32_t x) {
    x &= 0x3ffu;
    x = (x | (x << 16)) & 0x030000ffu;
    x = (x | (x << 8)) & 0x0300f00fu;
    x = (x | (x << 4)) & 0x030c30c3u;
    x = (x | (x << 2)) & 0x09249249u;
    return x;
}

// 10 bits per axis.  A zero, infinite or NaN extent, or a NaN centroid, quantises to 0 instead of an undefined
// conversion: the codes only shape the trees, never the result.
TRD uint32_t quantise(float c, float lo, float ext) {
    const float t = (ext > 0.0f && ext <= 3.4e38f) ? (c - lo) / ext * 1024.0f : 0.0f;
    if (!(t >= 0.0f)) return 0u;
    if (t >= 1023.0f) return 1023u;
    return (uint32_t)t;
}

// the last i in [0, n) with key(i) <= x, for keys that never decrease (0 if there is none)
template <typename KeyAt>
TRD uint32_t last_at_most(uint32_t n, uint32_t x, KeyAt key) {
    uint32_t lo = 0, hi = n;
    while (hi - lo > 1) {
        const uint32_t mid = (lo + hi) >> 1;
        if (key(mid) <= x) lo = mid;
        else hi = mid;
    }
    return lo;
}

// block-wide exclusive scan of one value per thread (blockDim.x a multiple of 32, at most 1024); returns the total in
// *total.  warp_sum holds 32 words; a caller that scans again must __syncthreads() first.
TRD uint32_t block_scan(uint32_t v, uint32_t* warp_sum, uint32_t* total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += y;
    }
    if (lane == 31) warp_sum[warp] = x;
    __syncthreads();
    if (warp == 0) {
        uint32_t s = lane < (int)(blockDim.x >> 5) ? warp_sum[lane] : 0u;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t y = __shfl_up_sync(0xffffffffu, s, o);
            if (lane >= o) s += y;
        }
        warp_sum[lane] = s;   // inclusive over warps
    }
    __syncthreads();
    const uint32_t excl = (warp ? warp_sum[warp - 1] : 0u) + x - v;
    *total = warp_sum[(blockDim.x >> 5) - 1];
    return excl;
}

// the empty box: lo > hi, and box_union with it leaves a box as it is
TRD void empty_box(float* lo, float* hi) {
    const float inf = __int_as_float(0x7f800000);
    lo[0] = lo[1] = lo[2] = inf;
    hi[0] = hi[1] = hi[2] = -inf;
}

// a triangle as the tris buffer holds it: three float4, w unused
struct Tri {
    float4 v[3];
};

// the vertices of indices [first, first + 3)
TRD Tri load_tri(const float* pos, const uint32_t* idx, uint32_t first) {
    Tri t;
#pragma unroll
    for (int k = 0; k < 3; k++) {
        const uint32_t v = __ldg(idx + first + k);
        t.v[k] = make_float4(__ldg(pos + (size_t)v * 3), __ldg(pos + (size_t)v * 3 + 1), __ldg(pos + (size_t)v * 3 + 2), 0.0f);
    }
    return t;
}

// the triangle's box as the host folds it: box_grow of each vertex into the empty box
TRD void tri_box(const Tri& t, float* lo, float* hi) {
    empty_box(lo, hi);
#pragma unroll
    for (int k = 0; k < 3; k++) {
        lo[0] = fminf(lo[0], t.v[k].x); hi[0] = fmaxf(hi[0], t.v[k].x);
        lo[1] = fminf(lo[1], t.v[k].y); hi[1] = fmaxf(hi[1], t.v[k].y);
        lo[2] = fminf(lo[2], t.v[k].z); hi[2] = fmaxf(hi[2], t.v[k].z);
    }
}

// box_union of the triangle's box into (lo, hi), as the host folds a leaf: a leaf's box is its triangles folded into
// the empty box
TRD void fold_tri(const Tri& t, float* lo, float* hi) {
    float tlo[3], thi[3];
    tri_box(t, tlo, thi);
#pragma unroll
    for (int k = 0; k < 3; k++) {
        lo[k] = fminf(fminf(lo[k], tlo[k]), thi[k]);
        hi[k] = fmaxf(fmaxf(hi[k], tlo[k]), thi[k]);
    }
}

// child `side`'s box: floats [6 side, 6 side + 6) of the node, lo then hi (the AccelNode layout)
TRD void store_box(AccelNode* n, int side, const float* lo, const float* hi) {
    float* b = reinterpret_cast<float*>(n) + side * 6;
    b[0] = lo[0]; b[1] = lo[1]; b[2] = lo[2];
    b[3] = hi[0]; b[4] = hi[1]; b[5] = hi[2];
}

// (lo, hi) united with the box of child `side`, which another thread stored: read through L2
TRD void union_child_box(const AccelNode* n, int side, float* lo, float* hi) {
    const float* b = reinterpret_cast<const float*>(n) + side * 6;
#pragma unroll
    for (int k = 0; k < 3; k++) {
        lo[k] = fminf(lo[k], __ldcg(b + k));
        hi[k] = fmaxf(hi[k], __ldcg(b + 3 + k));
    }
}

// One arrival of a bottom-up box pass at `node` from its child `side`: store (lo, hi) there, then count the arrival.  The
// first of the two arrivals returns false (the sibling's box is not there yet; the sibling's thread goes on from here).
// The second returns true, with (lo, hi) now the node's box.  fminf / fmaxf are exact, so the union does not depend on the
// arrival order (only the sign of a zero may).  The first fence publishes the box before the count, the second keeps the
// sibling's box from being read before the count.
TRD bool arrive(AccelNode* nodes, uint32_t* arrivals, int node, int side, float* lo, float* hi) {
    store_box(nodes + node, side, lo, hi);
    __threadfence();
    if (atomicAdd(&arrivals[node], 1u) == 0u) return false;
    __threadfence();
    union_child_box(nodes + node, side ^ 1, lo, hi);
    return true;
}

// build_tree's special roots (k_accel.cu): the empty tree, or one leaf wrapped in a root whose second box is empty; both
// children refer to leaf 0.  (lo, hi): the empty box, or the leaf's box.
TRD AccelNode special_root(const float* lo, const float* hi) {
    AccelNode r;
    store_box(&r, 0, lo, hi);
    empty_box(r.lo1, r.hi1);
    r.c0 = r.c1 = ~0;
    r.pad[0] = r.pad[1] = 0u;
    return r;
}

TRD TlasPrim make_tlas_prim(const float* lo, const float* hi, uint32_t blas_root, uint32_t tri_base, uint32_t keep) {
    TlasPrim p;
    for (int k = 0; k < 3; k++) {
        p.lo[k] = lo[k];
        p.hi[k] = hi[k];
    }
    p.blas_root = blas_root;
    p.tri_base = tri_base;
    p.keep = keep;
    p.pad[0] = p.pad[1] = p.pad[2] = 0u;
    return p;
}

// Stable LSD radix sort, one kRadixBits digit per pass.  The histogram counts every tile's digits, laid out digit-major,
// so the exclusive scan of hist is the first output slot of (digit, tile).  The scatter keeps the input order within a
// digit: stable.  The kernels are static: each translation unit that launches one has its own copy.
template <typename Key>
static __global__ void __launch_bounds__(kTile) radix_histogram_kernel(const Key* __restrict__ keys, uint32_t n, int shift,
                                                                       uint32_t* __restrict__ hist) {
    __shared__ uint32_t h[kRadix];
    h[threadIdx.x] = 0;
    __syncthreads();
    const uint32_t i = blockIdx.x * kTile + threadIdx.x;
    if (i < n) atomicAdd(&h[(uint32_t)(keys[i] >> shift) & (kRadix - 1)], 1u);
    __syncthreads();
    hist[(size_t)threadIdx.x * gridDim.x + blockIdx.x] = h[threadIdx.x];
}

template <typename Key>
static __global__ void __launch_bounds__(kTile) radix_scatter_kernel(const Key* __restrict__ keys, const uint32_t* __restrict__ vals, uint32_t n,
                                                                     int shift, const uint32_t* __restrict__ offset, Key* __restrict__ keys_out,
                                                                     uint32_t* __restrict__ vals_out) {
    __shared__ uint32_t digit[kTile];
    const uint32_t i = blockIdx.x * kTile + threadIdx.x;
    const Key key = i < n ? keys[i] : Key(0);
    const uint32_t d = i < n ? (uint32_t)(key >> shift) & (kRadix - 1) : 0xffffffffu;
    digit[threadIdx.x] = d;
    __syncthreads();
    if (i >= n) return;
    uint32_t rank = 0;
    for (uint32_t j = 0; j < threadIdx.x; j++) rank += digit[j] == d;
    const uint32_t dst = offset[(size_t)d * gridDim.x + blockIdx.x] + rank;
    keys_out[dst] = key;
    vals_out[dst] = vals[i];
}

}  // namespace trd
