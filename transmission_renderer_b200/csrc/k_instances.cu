// k_instances.cu — tr_update_instance_transforms: new transforms for a range of instances, in stream order.  The source is
// n packed 32-byte similarities (a device array of the caller's, or the context's staging copy of a host array); each
// thread moves one into the 48-byte tr_instance record with two 16-byte loads and two 16-byte stores, so primitive_id and
// material_id (bytes 32-39 of the record) are never touched.
#include "tr_internal.h"

namespace {

constexpr int kInstanceThreads = 256;

__global__ void __launch_bounds__(kInstanceThreads) instance_transforms_kernel(const float4* __restrict__ src, uint32_t n,
                                                                                tr_instance* __restrict__ dst) {
    const uint32_t i = blockIdx.x * kInstanceThreads + threadIdx.x;
    if (i >= n) return;
    const float4 a = __ldg(src + (size_t)i * 2), b = __ldg(src + (size_t)i * 2 + 1);
    float4* d = reinterpret_cast<float4*>(dst + i);
    d[0] = a;
    d[1] = b;
}

}  // namespace

namespace tr {

int32_t launch_instance_transforms(tr_ctx* c, uint32_t first, uint32_t n, const tr_packed_similarity* src) {
    instance_transforms_kernel<<<(n + kInstanceThreads - 1) / kInstanceThreads, kInstanceThreads, 0, c->stream>>>(
        reinterpret_cast<const float4*>(src), n, c->instances.as<tr_instance>() + first);
    count_launches(kInstanceTransformLaunches);
    TR_CUDA(cudaGetLastError());
    return TR_OK;
}

}  // namespace tr
