// k_textures.cu — tr_set_texture_async: a material image's level 0 (RGBA8) decoded into the sampler store and its mip chain
// built on the device, in stream order (sm_100a).
// Reference: load_texture_from_gltf + ImageManager::push_image (src/model_loading.rs:340-379): the loader uploads level 0
// and blits the rest of the chain on the GPU.  The filter and the rounding here are those of the Python ingest's CPU chain
// (scenes.make_mips), so that an image bound from level 0 is bit-equal to one bound through tr_set_texture with that chain:
//   * 2x2 box over the even-cropped source, in linear light (sRGB colour decoded, alpha and UNORM channels v / 255.0), in
//     float64, summed ((a + b) + c) + d — numpy's order for mean(axis=(1, 3)) — then halved twice (exact);
//   * every level rounded back to bytes as an RGBA8 image holds it: UNORM floor(clip(x) * 255 + 0.5), sRGB colour = the
//     number of the 255 encode thresholds <= x (texture_tables: bisection of the encode formula, libm pow on the host).
// Explicit __dadd_rn / __dmul_rn: nvcc must not contract the filter into FMAs (numpy does not).
// Layout of an image's allocation: the RGBA32F store the samplers read (TexDesc.off), then the RGBA8 bytes of every level at
// the same texel offsets.  The bytes are the next level's source and nothing else reads them.
// One launch per level.  Level 0: 4 B in, 16 B out per texel.  Level k: 16 B in (four source texels), 4 + 16 B out.
#include <math.h>
#include <string.h>

#include "tr_internal.h"

namespace {

constexpr int kThreads = 256;

// sRGB8 -> linear in double (R8G8B8A8_SRGB decode); the store rounds it to float once
double srgb8_to_linear64(int v) {
    const double x = (double)v / 255.0;
    return x <= 0.04045 ? x / 12.92 : pow((x + 0.055) / 1.055, 2.4);
}

// scenes.srgb_encode of one value (clip, OETF, floor(s * 255 + 0.5)), libm pow
int srgb_encode_byte(double x) {
    x = x < 0.0 ? 0.0 : (x > 1.0 ? 1.0 : x);
    const double s = x <= 0.0031308 ? x * 12.92 : 1.055 * pow(x, 1.0 / 2.4) - 0.055;
    return (int)floor(s * 255.0 + 0.5);
}

tr::TexTables build_tables() {
    tr::TexTables t;
    for (int v = 0; v < 256; v++) {
        t.dec64[0][v] = srgb8_to_linear64(v);
        t.dec64[1][v] = (double)v / 255.0;
        t.dec32[0][v] = (float)t.dec64[0][v];
        t.dec32[1][v] = (float)v / 255.0f;   // alpha stays linear in the sRGB formats
    }
    // encode[k - 1] = the smallest double x in [0, 1] whose byte is >= k: bisection on the bit patterns, which order the
    // non-negative doubles as their values do
    for (int k = 1; k < 256; k++) {
        uint64_t lo = 0, hi;   // byte(lo) < k <= byte(hi)
        const double one = 1.0;
        memcpy(&hi, &one, 8);
        while (hi - lo > 1) {
            const uint64_t mid = lo + (hi - lo) / 2;
            double x;
            memcpy(&x, &mid, 8);
            if (srgb_encode_byte(x) >= k) hi = mid;
            else lo = mid;
        }
        memcpy(&t.encode[k - 1], &hi, 8);
    }
    t.encode[255] = 2.0;   // above every filtered value: the search below never passes it
    return t;
}

__device__ __forceinline__ void load_tables(const tr::TexTables* __restrict__ g, tr::TexTables& s) {
    const uint4* src = reinterpret_cast<const uint4*>(g);
    uint4* dst = reinterpret_cast<uint4*>(&s);
    for (uint32_t i = threadIdx.x; i < sizeof(tr::TexTables) / 16; i += blockDim.x) dst[i] = src[i];
    __syncthreads();
}

__device__ __forceinline__ float4 decode(const tr::TexTables& t, uchar4 b, int colour) {
    return make_float4(t.dec32[colour][b.x], t.dec32[colour][b.y], t.dec32[colour][b.z], t.dec32[1][b.w]);
}

// level 0: the RGBA8 bytes (copied in front of this launch) into the store
__global__ void __launch_bounds__(kThreads) texture_level0_kernel(const tr::TexTables* __restrict__ tables,
                                                                  const uchar4* __restrict__ bytes, float4* __restrict__ store,
                                                                  uint32_t n, int colour) {
    __shared__ tr::TexTables t;
    load_tables(tables, t);
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
        __stcs(store + i, decode(t, __ldcs(bytes + i), colour));
}

__device__ __forceinline__ double box(const double* dec, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    return __dmul_rn(__dadd_rn(__dadd_rn(__dadd_rn(dec[a], dec[b]), dec[c]), dec[d]), 0.25);
}

__device__ __forceinline__ uint32_t unorm_byte(double x) {   // floor(clip(x) * 255 + 0.5)
    x = fmin(fmax(x, 0.0), 1.0);
    return (uint32_t)floor(__dadd_rn(__dmul_rn(x, 255.0), 0.5));
}

__device__ __forceinline__ uint32_t srgb_byte(const double* encode, double x) {   // thresholds <= x (encode[255] = 2)
    uint32_t k = 0;
#pragma unroll
    for (uint32_t s = 128; s; s >>= 1)
        if (encode[k + s - 1] <= x) k += s;
    return k;
}

// level k from the bytes of level k - 1 (sw x sh, both >= 2): bytes and store of level k (w x h = sw / 2 x sh / 2)
__global__ void __launch_bounds__(kThreads) texture_level_kernel(const tr::TexTables* __restrict__ tables,
                                                                 const uchar4* __restrict__ src, uint32_t sw,
                                                                 uchar4* __restrict__ bytes, float4* __restrict__ store,
                                                                 uint32_t w, uint32_t h, int colour) {
    __shared__ tr::TexTables t;
    load_tables(tables, t);
    const double* dc = t.dec64[colour];
    const double* da = t.dec64[1];
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < w * h; i += gridDim.x * blockDim.x) {
        const uint32_t y = i / w, x = i - y * w;
        const uchar4* row = src + (size_t)(2 * y) * sw + 2 * x;
        const uchar4 a = row[0], b = row[1], c = row[sw], d = row[sw + 1];
        const double r = box(dc, a.x, b.x, c.x, d.x), g = box(dc, a.y, b.y, c.y, d.y), bl = box(dc, a.z, b.z, c.z, d.z);
        const double al = box(da, a.w, b.w, c.w, d.w);
        uchar4 o;
        o.x = (unsigned char)(colour == 0 ? srgb_byte(t.encode, r) : unorm_byte(r));
        o.y = (unsigned char)(colour == 0 ? srgb_byte(t.encode, g) : unorm_byte(g));
        o.z = (unsigned char)(colour == 0 ? srgb_byte(t.encode, bl) : unorm_byte(bl));
        o.w = (unsigned char)unorm_byte(al);
        bytes[i] = o;
        __stcs(store + i, decode(t, o, colour));
    }
}

uint32_t grid_for(size_t n, int sm_count) {   // a few blocks per SM: each block loads the 8 KB of tables once
    size_t blocks = (n + kThreads - 1) / kThreads;
    const size_t cap = (size_t)sm_count * 8;
    if (blocks > cap) blocks = cap;
    return blocks ? (uint32_t)blocks : 1u;
}

}  // namespace

namespace tr {

const TexTables& texture_tables() {
    static const TexTables t = build_tables();
    return t;
}

int32_t launch_texture_chain(const TexTables* d_tables, const trd::TexDesc& d, uint8_t* chain, int sm_count, cudaStream_t s) {
    const int colour = d.srgb ? 0 : 1;
    float4* store = const_cast<float4*>(d.base);
    uchar4* bytes = reinterpret_cast<uchar4*>(chain);
    const size_t n0 = (size_t)d.w * d.h;
    texture_level0_kernel<<<grid_for(n0, sm_count), kThreads, 0, s>>>(d_tables, bytes, store, (uint32_t)n0, colour);
    for (uint32_t l = 1; l < d.levels; l++) {
        const uint32_t sw = d.w >> (l - 1) ? d.w >> (l - 1) : 1u;
        const uint32_t w = d.w >> l ? d.w >> l : 1u, h = d.h >> l ? d.h >> l : 1u;
        texture_level_kernel<<<grid_for((size_t)w * h, sm_count), kThreads, 0, s>>>(
            d_tables, bytes + d.off[l - 1], sw, bytes + d.off[l], store + d.off[l], w, h, colour);
    }
    count_launches((int)d.levels);
    TR_CUDA(cudaGetLastError());
    return TR_OK;
}

}  // namespace tr
