// tr_comm.cu — multi-GPU plumbing: one context per rank/GPU, image bands (SURVEY.md 8e).
//
// The reference is single-GPU (one VkQueue, src/main.rs:243); band sharding is new work defined by
// the north star.  Between K4 (opaque bands) and K5 (mips) every rank needs the WHOLE mip-0 frame,
// because the refraction fetch of glam-pbr lib.rs:330-337 reads arbitrary texels.  Two ways:
//   (a) NCCL all-gather, in place in the full-frame buffer (baseline);
//   (b) peer stores: K4's odd lanes write the band straight into every peer's mip 0 over
//       NVLink (CUDA IPC mappings), so the exchange overlaps shading tile by tile; what is left is a
//       cross-GPU barrier, done with release/acquire flag words in the same peer memory (no NCCL call
//       in the frame loop).
// NCCL is resolved at run time (dlsym on the already-loaded libnccl.so.2 of the host process,
// e.g. torch's, else dlopen) so single-GPU users need no NCCL at all.
#include <dlfcn.h>
#include <string.h>

#include "tr_internal.h"

namespace tr {

namespace {
typedef struct { char internal[128]; } nccl_unique_id;
typedef int (*fn_get_unique_id)(nccl_unique_id*);
typedef int (*fn_comm_init_rank)(void**, int, nccl_unique_id, int);
typedef int (*fn_comm_destroy)(void*);
typedef int (*fn_all_gather)(const void*, void*, size_t, int, void*, cudaStream_t);
typedef int (*fn_all_reduce)(const void*, void*, size_t, int, int, void*, cudaStream_t);
typedef int (*fn_broadcast)(const void*, void*, size_t, int, int, void*, cudaStream_t);
typedef int (*fn_group)(void);
typedef const char* (*fn_error_string)(int);

struct NcclApi {
    bool loaded = false, ok = false;
    fn_get_unique_id get_unique_id = nullptr;
    fn_comm_init_rank comm_init_rank = nullptr;
    fn_comm_destroy comm_destroy = nullptr;
    fn_all_gather all_gather = nullptr;
    fn_all_reduce all_reduce = nullptr;
    fn_broadcast broadcast = nullptr;
    fn_group group_start = nullptr, group_end = nullptr;
    fn_error_string error_string = nullptr;
} g_nccl;

constexpr int kNcclUint8 = 1, kNcclInt32 = 2, kNcclSum = 0;

bool load_nccl() {
    if (g_nccl.loaded) return g_nccl.ok;
    g_nccl.loaded = true;
    void* h = RTLD_DEFAULT;
    if (!dlsym(h, "ncclAllGather")) {
        h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
        if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
        if (!h) return false;
    }
    g_nccl.get_unique_id = (fn_get_unique_id)dlsym(h, "ncclGetUniqueId");
    g_nccl.comm_init_rank = (fn_comm_init_rank)dlsym(h, "ncclCommInitRank");
    g_nccl.comm_destroy = (fn_comm_destroy)dlsym(h, "ncclCommDestroy");
    g_nccl.all_gather = (fn_all_gather)dlsym(h, "ncclAllGather");
    g_nccl.all_reduce = (fn_all_reduce)dlsym(h, "ncclAllReduce");
    g_nccl.broadcast = (fn_broadcast)dlsym(h, "ncclBroadcast");
    g_nccl.group_start = (fn_group)dlsym(h, "ncclGroupStart");
    g_nccl.group_end = (fn_group)dlsym(h, "ncclGroupEnd");
    g_nccl.error_string = (fn_error_string)dlsym(h, "ncclGetErrorString");
    g_nccl.ok = g_nccl.get_unique_id && g_nccl.comm_init_rank && g_nccl.comm_destroy && g_nccl.all_gather &&
                g_nccl.all_reduce && g_nccl.broadcast && g_nccl.group_start && g_nccl.group_end;
    return g_nccl.ok;
}

int32_t nccl_fail(const char* what, int rc) {
    return fail(TR_ERR_NCCL, "%s: %s", what, g_nccl.error_string ? g_nccl.error_string(rc) : "NCCL error");
}
}  // namespace

void band_of(const tr_ctx* c, int r, uint32_t* y0, uint32_t* y1) {
    if (c->band_bounds.size() == (size_t)c->n_ranks + 1) {  // caller-balanced bands (tr_set_bands)
        *y0 = c->band_bounds[r];
        *y1 = c->band_bounds[r + 1];
        return;
    }
    *y0 = (uint32_t)(((uint64_t)r * c->height) / c->n_ranks);
    *y1 = (uint32_t)(((uint64_t)(r + 1) * c->height) / c->n_ranks);
}

namespace {
struct PeerFlags {
    uint32_t* p[kMaxPeers];
};
// Barrier over NVLink peer memory: thread t tells rank t "rank `rank` has reached epoch e" with a release store into
// that rank's words, then waits (acquire loads on its own words) until rank t has said the same.  The opaque pass's peer
// stores of this rank completed with its kernel, i.e. before this kernel started, so a rank that leaves the barrier
// sees every band in its own mip 0.
__global__ void peer_barrier_kernel(PeerFlags f, int rank, int n_ranks, uint32_t epoch) {
    const int t = threadIdx.x;
    if (t >= n_ranks) return;
    __threadfence_system();
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(f.p[t] + rank), "r"(epoch) : "memory");
    uint32_t v;
    do {
        asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(f.p[rank] + t) : "memory");
    } while ((int32_t)(v - epoch) < 0);
}
}  // namespace

// cross-GPU barrier on the context's stream: flags in peer memory when the peer mappings exist, else a 4-byte all-reduce
int32_t comm_barrier(tr_ctx* c) {
    if (c->n_ranks <= 1) return TR_OK;
    if (c->peers_attached) {
        PeerFlags f{};
        for (int r = 0; r < c->n_ranks; r++) f.p[r] = c->peer_flags[r];
        peer_barrier_kernel<<<1, 32, 0, c->stream>>>(f, c->rank, c->n_ranks, ++c->barrier_epoch);
        count_launches(1);
        TR_CUDA(cudaGetLastError());
        return TR_OK;
    }
    if (!c->nccl_comm) return fail(TR_ERR_STATE, "communicator not initialised (tr_comm_init)");
    uint32_t* scratch = c->mip_counter.as<uint32_t>() + 2;
    int rc = g_nccl.all_reduce(scratch, scratch, 1, kNcclInt32, kNcclSum, c->nccl_comm, c->stream);
    if (rc) return nccl_fail("ncclAllReduce", rc);
    return TR_OK;
}

int32_t comm_allgather_opaque(tr_ctx* c) {
    if (c->n_ranks <= 1) return TR_OK;
    if (!c->nccl_comm) return fail(TR_ERR_STATE, "tr_allgather_opaque: communicator not initialised (tr_comm_init)");
    // peer-store path: bands are already in place everywhere once every rank's K4 has retired
    if (c->peers_attached) return comm_barrier(c);
    uint8_t* mip0 = reinterpret_cast<uint8_t*>(c->pyramid.as<uint2>() + c->level_off[0]);
    const size_t row = (size_t)c->width * 8;
    if (c->band_bounds.empty() && c->height % c->n_ranks == 0) {
        const size_t count = (size_t)(c->height / c->n_ranks) * row;
        int rc = g_nccl.all_gather(mip0 + (size_t)c->rank * count, mip0, count, kNcclUint8, c->nccl_comm, c->stream);
        if (rc) return nccl_fail("ncclAllGather", rc);
    } else {
        int rc = g_nccl.group_start();
        if (rc) return nccl_fail("ncclGroupStart", rc);
        for (int r = 0; r < c->n_ranks; r++) {
            uint32_t y0, y1;
            band_of(c, r, &y0, &y1);
            uint8_t* p = mip0 + (size_t)y0 * row;
            rc = g_nccl.broadcast(p, p, (size_t)(y1 - y0) * row, kNcclUint8, r, c->nccl_comm, c->stream);
            if (rc) return nccl_fail("ncclBroadcast", rc);
        }
        rc = g_nccl.group_end();
        if (rc) return nccl_fail("ncclGroupEnd", rc);
    }
    return TR_OK;
}

void comm_release(tr_ctx* c) {
    if (c->peers_attached) {
        for (int r = 0; r < c->n_ranks; r++)
            if (r != c->rank && c->peer_mip0[r]) cudaIpcCloseMemHandle(c->peer_mip0[r]);
        c->peers_attached = false;
    }
    if (c->nccl_comm && g_nccl.ok) g_nccl.comm_destroy(c->nccl_comm);
    c->nccl_comm = nullptr;
}

}  // namespace tr

using namespace tr;

extern "C" {

int32_t tr_comm_unique_id(uint8_t id[TR_NCCL_UNIQUE_ID_BYTES]) {
    if (!id) return fail(TR_ERR_INVALID_ARG, "tr_comm_unique_id: null");
    if (!load_nccl()) return fail(TR_ERR_NCCL, "NCCL library not found (libnccl.so.2)");
    nccl_unique_id u;
    int rc = g_nccl.get_unique_id(&u);
    if (rc) return nccl_fail("ncclGetUniqueId", rc);
    memcpy(id, &u, sizeof(u));
    return TR_OK;
}

int32_t tr_comm_init(tr_ctx* c, const uint8_t id[TR_NCCL_UNIQUE_ID_BYTES], int32_t rank, int32_t n_ranks) {
    if (!c || !id) return fail(TR_ERR_INVALID_ARG, "tr_comm_init: null");
    if (n_ranks < 1 || n_ranks > kMaxPeers || rank < 0 || rank >= n_ranks)
        return fail(TR_ERR_INVALID_ARG, "tr_comm_init: rank %d of %d (at most %d ranks)", rank, n_ranks, kMaxPeers);
    TR_NOT_GROUPED(c, "tr_comm_init", "the group's bands (tr_group_set_bands); a group needs no communicator");
    TR_CUDA(cudaSetDevice(c->device));
    c->rank = rank;
    c->n_ranks = n_ranks;
    c->band_bounds.clear();
    uint32_t y0, y1;
    band_of(c, rank, &y0, &y1);
    c->band_y0 = y0;
    c->band_y1 = y1;
    if (n_ranks == 1) return TR_OK;
    if (!load_nccl()) return fail(TR_ERR_NCCL, "NCCL library not found (libnccl.so.2)");
    nccl_unique_id u;
    memcpy(&u, id, sizeof(u));
    int rc = g_nccl.comm_init_rank(&c->nccl_comm, n_ranks, u, rank);
    if (rc) return nccl_fail("ncclCommInitRank", rc);
    return TR_OK;
}

int32_t tr_comm_destroy(tr_ctx* c) {
    if (!c) return TR_OK;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    comm_release(c);
    c->rank = 0;
    c->n_ranks = 1;
    c->band_bounds.clear();
    c->band_y0 = 0;
    c->band_y1 = c->height;
    return TR_OK;
}

int32_t tr_set_bands(tr_ctx* c, const uint32_t* bounds, uint32_t n_bounds) {
    if (!c || !bounds) return fail(TR_ERR_INVALID_ARG, "tr_set_bands: null");
    TR_NOT_GROUPED(c, "tr_set_bands", "tr_group_set_bands");
    if (n_bounds != (uint32_t)c->n_ranks + 1) return fail(TR_ERR_INVALID_ARG, "tr_set_bands: %u boundaries for %d ranks", n_bounds, c->n_ranks);
    if (bounds[0] != 0 || bounds[c->n_ranks] != c->height) return fail(TR_ERR_INVALID_ARG, "tr_set_bands: the bands must cover rows [0, %u)", c->height);
    for (int r = 0; r < c->n_ranks; r++)
        if (bounds[r] >= bounds[r + 1]) return fail(TR_ERR_INVALID_ARG, "tr_set_bands: band %d is empty", r);
    c->band_bounds.assign(bounds, bounds + n_bounds);
    c->band_y0 = bounds[c->rank];
    c->band_y1 = bounds[c->rank + 1];
    return TR_OK;
}

int32_t tr_peer_export(tr_ctx* c, uint8_t handle[TR_IPC_HANDLE_BYTES]) {
    if (!c || !handle) return fail(TR_ERR_INVALID_ARG, "tr_peer_export: null");
    TR_CUDA(cudaSetDevice(c->device));
    static_assert(sizeof(cudaIpcMemHandle_t) == TR_IPC_HANDLE_BYTES, "IPC handle size");
    // the barrier words behind the pyramid start at epoch 0, before any peer can map them
    TR_CUDA(cudaStreamSynchronize(c->stream));
    TR_CUDA(cudaMemset(c->pyramid.as<unsigned char>() + c->barrier_flags_offset, 0, 256));
    c->barrier_epoch = 0;
    cudaIpcMemHandle_t h;
    TR_CUDA(cudaIpcGetMemHandle(&h, c->pyramid.p));
    memcpy(handle, &h, sizeof(h));
    return TR_OK;
}

int32_t tr_peer_attach(tr_ctx* c, int32_t rank, int32_t n_ranks, const uint8_t* handles) {
    if (!c || !handles) return fail(TR_ERR_INVALID_ARG, "tr_peer_attach: null");
    TR_NOT_GROUPED(c, "tr_peer_attach", "tr_group_frame, whose members store into each other's frames directly");
    if (rank != c->rank || n_ranks != c->n_ranks) return fail(TR_ERR_STATE, "tr_peer_attach: call tr_comm_init first with the same rank/size");
    TR_CUDA(cudaSetDevice(c->device));
    for (int r = 0; r < n_ranks; r++) {
        if (r == rank) {
            c->peer_mip0[r] = c->pyramid.as<uint2>() + c->level_off[0];
            c->peer_flags[r] = reinterpret_cast<uint32_t*>(c->pyramid.as<unsigned char>() + c->barrier_flags_offset);
            continue;
        }
        cudaIpcMemHandle_t h;
        memcpy(&h, handles + (size_t)r * TR_IPC_HANDLE_BYTES, sizeof(h));
        void* p = nullptr;
        TR_CUDA(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
        c->peer_mip0[r] = reinterpret_cast<uint2*>(p) + c->level_off[0];
        c->peer_flags[r] = reinterpret_cast<uint32_t*>(reinterpret_cast<unsigned char*>(p) + c->barrier_flags_offset);
    }
    c->peers_attached = true;
    return TR_OK;
}

}  // extern "C"
