// tr_group.cu — several contexts of ONE host thread rendering the bands of one frame (include/tr_abi.h, "Multi-GPU in one
// process").  The reference's host is one thread with one queue (src/main.rs:243, 1290-1294); the multi-process band path
// (tr_comm.cu) needs a process per GPU.  A group runs the same band split and the same fused peer-store exchange from one
// thread:
//
//   * exchange: member k's opaque pass (K4) stores its band into every member's mip 0 (ShadeLaunch::opaque[], filled from
//     the group in tr_api.cu shade_opaque).  The bases are plain device pointers, on a peer device or on the same one.
//   * ordering: CUDA events only.  A spin barrier (tr_comm.cu peer_barrier_kernel) waits for a flag another rank sets; with
//     one enqueuing thread it hangs the GPU as soon as the enqueue of a later member blocks (a chunk rebuild, a buffer
//     growing, the synchronous copy of an upload).  tr_group_frame makes two passes over the members:
//       front  r: timer mark, K2 | K1 + K3, join; wait for every other member's BACK event of the previous group frame
//                 (its K6 no longer samples its mip 0, which r's K4 is about to write); K4; record r's FRONT event
//       back   r: wait for every other member's FRONT event of this frame (every band is in r's mip 0); K5, K6; record
//                 r's BACK event; K7
//   * replication (tr_group_replicate_scene): the source records its REPLICA event; each destination d waits for it, copies
//     the scene on its own stream (tr_api.cu replicate_scene: copy engines only, from a peer device or the same one) and
//     records d's REPLICA event; then the source waits for every destination's REPLICA event, so that a later upload to
//     the source cannot overwrite what a copy is still reading.  A frame a destination enqueued before the call reads the
//     old scene, its next frame the new one.
//     Every wait, the frame's and the replication's, names an event whose record call this thread has already made (the
//     first frame's waits name events never recorded, which CUDA treats as complete), so no enqueued work depends on work
//     not yet enqueued: nothing can deadlock.
#include <string.h>

#include <new>

#include "tr_internal.h"

using namespace tr;

namespace {

int32_t set_device(const tr_ctx* c) {
    TR_CUDA(cudaSetDevice(c->device));
    return TR_OK;
}

// Distinct devices store into each other's frames: peer access both ways.  "Already enabled" (by torch, or an earlier
// group) is success; access stays enabled after the group, since the host process may rely on it.  Stream-ordered pool
// memory does not follow cudaDeviceEnablePeerAccess: the images tr_set_texture_async allocates from each device's default
// pool (tr_api.cu ensure_texture), which tr_group_replicate_scene copies across devices, so that pool is opened to the
// other device too (read and write, both ways; it stays open, like peer access).
int32_t enable_peer_access(int a, int b) {
    int ab = 0, ba = 0;
    TR_CUDA(cudaDeviceCanAccessPeer(&ab, a, b));
    TR_CUDA(cudaDeviceCanAccessPeer(&ba, b, a));
    if (!ab || !ba)
        return fail(TR_ERR_UNSUPPORTED, "tr_group_create: devices %d and %d have no peer access in both directions; a group "
                                        "stores every band into every member's frame directly", a, b);
    for (int k = 0; k < 2; k++) {
        const int from = k ? b : a, to = k ? a : b;
        TR_CUDA(cudaSetDevice(from));
        const cudaError_t e = cudaDeviceEnablePeerAccess(to, 0);
        if (e == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();   // clears it
        else if (e != cudaSuccess)
            return fail(TR_ERR_CUDA, "tr_group_create: cudaDeviceEnablePeerAccess(%d -> %d): %s", from, to, cudaGetErrorString(e));
        cudaMemPool_t pool;
        TR_CUDA(cudaDeviceGetDefaultMemPool(&pool, to));
        cudaMemAccessDesc access{};
        access.location.type = cudaMemLocationTypeDevice;
        access.location.id = from;
        access.flags = cudaMemAccessFlagsProtReadWrite;
        TR_CUDA(cudaMemPoolSetAccess(pool, &access, 1));   // `from` reads and writes `to`'s pool
    }
    return TR_OK;
}

// member k: rank k of n, equal-row bands (band_of), or the caller's boundaries
void set_rank(tr_ctx* c, int rank, int n) {
    c->rank = rank;
    c->n_ranks = n;
    band_of(c, rank, &c->band_y0, &c->band_y1);
}

int32_t sync_members(tr_group* g) {
    for (int k = 0; k < g->n; k++) {
        tr_ctx* c = g->members[k];
        TR_TRY(set_device(c));
        TR_CUDA(cudaStreamSynchronize(c->stream));
        if (c->copy_stream) TR_CUDA(cudaStreamSynchronize(c->copy_stream));
    }
    return TR_OK;
}

void destroy_events(tr_group* g) {
    for (int k = 0; k < g->n; k++) {
        cudaSetDevice(g->members[k]->device);
        if (g->ev_front[k]) cudaEventDestroy(g->ev_front[k]);
        if (g->ev_back[k]) cudaEventDestroy(g->ev_back[k]);
        if (g->ev_replica[k]) cudaEventDestroy(g->ev_replica[k]);
        g->ev_front[k] = g->ev_back[k] = g->ev_replica[k] = nullptr;
    }
}

}  // namespace

extern "C" {

int32_t tr_group_create(tr_ctx* const* ctxs, uint32_t n, tr_group** out_group) {
    if (!ctxs || !out_group) return fail(TR_ERR_INVALID_ARG, "tr_group_create: null argument");
    *out_group = nullptr;
    if (n == 0 || n > (uint32_t)kMaxPeers) return fail(TR_ERR_INVALID_ARG, "tr_group_create: %u members (1..%d)", n, kMaxPeers);
    for (uint32_t k = 0; k < n; k++) {
        const tr_ctx* c = ctxs[k];
        if (!c) return fail(TR_ERR_INVALID_ARG, "tr_group_create: member %u is null", k);
        if (c->height < n) return fail(TR_ERR_INVALID_ARG, "tr_group_create: %u rows for %u bands", c->height, n);
        for (uint32_t j = 0; j < k; j++)
            if (ctxs[j] == c) return fail(TR_ERR_INVALID_ARG, "tr_group_create: members %u and %u are the same context", j, k);
        if (c->width != ctxs[0]->width || c->height != ctxs[0]->height)
            return fail(TR_ERR_INVALID_ARG, "tr_group_create: member %u is %ux%u, member 0 %ux%u", k, c->width, c->height,
                        ctxs[0]->width, ctxs[0]->height);
        if (c->group) return fail(TR_ERR_STATE, "tr_group_create: member %u is in another group (tr_group_destroy it first)", k);
        if (c->nccl_comm || c->n_ranks > 1)
            return fail(TR_ERR_STATE, "tr_group_create: member %u is a rank of a communicator (tr_comm_destroy first)", k);
        if (c->peers_attached) return fail(TR_ERR_STATE, "tr_group_create: member %u has peer mappings (tr_comm_destroy first)", k);
    }
    for (uint32_t k = 0; k < n; k++)
        for (uint32_t j = 0; j < k; j++)
            if (ctxs[j]->device != ctxs[k]->device) TR_TRY(enable_peer_access(ctxs[j]->device, ctxs[k]->device));
    tr_group* g = new (std::nothrow) tr_group();
    if (!g) return fail(TR_ERR_OOM, "tr_group_create: host allocation failed");
    g->n = (int)n;
    int32_t st = TR_OK;
    for (uint32_t k = 0; k < n && st == TR_OK; k++) {
        tr_ctx* c = ctxs[k];
        g->members[k] = c;
        st = set_device(c);
        // a frame still in flight samples its own mip 0, which the other members' first opaque passes will write
        if (st == TR_OK && cudaStreamSynchronize(c->stream) != cudaSuccess) st = fail(TR_ERR_CUDA, "tr_group_create: member %u's stream failed", k);
        if (st == TR_OK && (cudaEventCreateWithFlags(&g->ev_front[k], cudaEventDisableTiming) != cudaSuccess ||
                            cudaEventCreateWithFlags(&g->ev_back[k], cudaEventDisableTiming) != cudaSuccess ||
                            cudaEventCreateWithFlags(&g->ev_replica[k], cudaEventDisableTiming) != cudaSuccess))
            st = fail(TR_ERR_CUDA, "tr_group_create: cudaEventCreate failed");
    }
    if (st != TR_OK) {
        destroy_events(g);
        delete g;
        return st;
    }
    for (uint32_t k = 0; k < n; k++) {
        tr_ctx* c = ctxs[k];
        c->band_bounds.clear();
        set_rank(c, (int)k, (int)n);
        c->group = g;
    }
    *out_group = g;
    return TR_OK;
}

int32_t tr_group_destroy(tr_group* g) {
    if (!g) return TR_OK;
    const int32_t st = sync_members(g);   // a member's opaque pass may still be storing into another's frame
    destroy_events(g);
    for (int k = 0; k < g->n; k++) {
        tr_ctx* c = g->members[k];
        c->group = nullptr;
        c->band_bounds.clear();
        c->rank = 0;
        c->n_ranks = 1;
        c->band_y0 = 0;
        c->band_y1 = c->height;
    }
    delete g;
    return st;
}

int32_t tr_group_set_bands(tr_group* g, const uint32_t* bounds, uint32_t n_bounds) {
    if (!g || !bounds) return fail(TR_ERR_INVALID_ARG, "tr_group_set_bands: null");
    const uint32_t h = g->members[0]->height;
    if (n_bounds != (uint32_t)g->n + 1) return fail(TR_ERR_INVALID_ARG, "tr_group_set_bands: %u boundaries for %d members", n_bounds, g->n);
    if (bounds[0] != 0 || bounds[g->n] != h) return fail(TR_ERR_INVALID_ARG, "tr_group_set_bands: the bands must cover rows [0, %u)", h);
    for (int r = 0; r < g->n; r++)
        if (bounds[r] >= bounds[r + 1]) return fail(TR_ERR_INVALID_ARG, "tr_group_set_bands: band %d is empty", r);
    for (int k = 0; k < g->n; k++) {
        tr_ctx* c = g->members[k];
        c->band_bounds.assign(bounds, bounds + n_bounds);
        set_rank(c, k, g->n);
    }
    return TR_OK;
}

int32_t tr_group_resize(tr_group* g, uint32_t width, uint32_t height) {
    if (!g) return fail(TR_ERR_INVALID_ARG, "tr_group_resize: null");
    if (width == 0 || height == 0) return fail(TR_ERR_INVALID_ARG, "tr_group_resize: empty framebuffer");
    if (height < (uint32_t)g->n) return fail(TR_ERR_INVALID_ARG, "tr_group_resize: %u rows for %d bands", height, g->n);
    TR_TRY(sync_members(g));   // every member's frame buffers may be reallocated, and every member stores into all of them
    for (int k = 0; k < g->n; k++) {
        tr_ctx* c = g->members[k];
        TR_TRY(set_device(c));
        TR_TRY(resize_frame(c, width, height));   // rank k of n keeps an equal-rows band; the mip-0 bases are re-read per frame
    }
    return TR_OK;
}

int32_t tr_group_frame(tr_group* g, const tr_frame_params* params) {
    if (!g || !params) return fail(TR_ERR_INVALID_ARG, "tr_group_frame: null");
    for (int k = 0; k < g->n; k++)   // refuse bad parameters before anything is enqueued
        TR_TRY(check_pc(g->members[k], &params[k].push_constants, "tr_group_frame"));
    for (int r = 0; r < g->n; r++) {   // front: everything up to K4; K4 waits until no member still samples its frame
        tr_ctx* c = g->members[r];
        TR_TRY(set_device(c));
        TR_TRY(frame_front(c, &params[r]));
        for (int k = 0; k < g->n; k++)
            if (k != r) TR_CUDA(cudaStreamWaitEvent(c->stream, g->ev_back[k], 0));
        TR_TRY(shade_opaque(c, &params[r].push_constants));
        TR_CUDA(cudaEventRecord(g->ev_front[r], c->stream));
    }
    for (int r = 0; r < g->n; r++) {   // back: the exchange is complete once every member's K4 has retired
        tr_ctx* c = g->members[r];
        TR_TRY(set_device(c));
        pass_begin(c, P_GATHER);
        for (int k = 0; k < g->n; k++)
            if (k != r) TR_CUDA(cudaStreamWaitEvent(c->stream, g->ev_front[k], 0));
        pass_end(c, P_GATHER);
        TR_TRY(frame_back(c, &params[r], g->ev_back[r]));
    }
    return TR_OK;
}

int32_t tr_group_replicate_scene(tr_group* g, uint32_t source, uint64_t* addresses) {
    if (!g) return fail(TR_ERR_INVALID_ARG, "tr_group_replicate_scene: null");
    if (source >= (uint32_t)g->n) return fail(TR_ERR_INVALID_ARG, "tr_group_replicate_scene: source %u of %d members", source, g->n);
    tr_ctx* s = g->members[source];
    if (!s->mesh_pos.p) return fail(TR_ERR_STATE, "tr_group_replicate_scene: member %u has no mesh (tr_set_mesh)", source);
    int32_t st = TR_OK;
    if (g->n > 1) {
        TR_TRY(set_device(s));
        TR_CUDA(cudaEventRecord(g->ev_replica[source], s->stream));
        int issued = 0;   // destinations [0, issued) may have copies in flight that read the source
        for (int k = 0; k < g->n && st == TR_OK; k++) {
            if (k == (int)source) continue;
            tr_ctx* d = g->members[k];
            st = set_device(d);
            if (st == TR_OK && cudaStreamWaitEvent(d->stream, g->ev_replica[source], 0) != cudaSuccess)
                st = fail(TR_ERR_CUDA, "tr_group_replicate_scene: member %d cannot wait for the source", k);
            if (st != TR_OK) break;
            st = replicate_scene(d, s);
            issued = k + 1;
            if (cudaEventRecord(g->ev_replica[k], d->stream) != cudaSuccess && st == TR_OK)
                st = fail(TR_ERR_CUDA, "tr_group_replicate_scene: cudaEventRecord on member %d failed", k);
        }
        // later work on the source (an upload into a buffer a copy is still reading) waits for every copy
        TR_TRY(set_device(s));
        for (int k = 0; k < issued; k++)
            if (k != (int)source) TR_CUDA(cudaStreamWaitEvent(s->stream, g->ev_replica[k], 0));
    }
    if (addresses)
        for (int k = 0; k < g->n; k++) {
            const tr_ctx* m = g->members[k];
            addresses[k] = m->accel_blas_valid && m->accel_tlas_valid ? (uint64_t)(uintptr_t)m->accel_tlas.p : 0;
        }
    return st;
}

int32_t tr_group_sync(tr_group* g) {
    if (!g) return fail(TR_ERR_INVALID_ARG, "tr_group_sync: null");
    for (int k = 0; k < g->n; k++) TR_TRY(tr_sync(g->members[k]));
    return TR_OK;
}

int32_t tr_group_read_srgb8(tr_group* g, uint8_t* rgba8) {
    if (!g || !rgba8) return fail(TR_ERR_INVALID_ARG, "tr_group_read_srgb8: null");
    for (int k = 0; k < g->n; k++)
        if (!g->members[k]->srgb_valid) return fail(TR_ERR_STATE, "tr_group_read_srgb8: member %d has not tonemapped a frame", k);
    for (int k = 0; k < g->n; k++) {   // one copy per band, each behind its member's frame, as tr_read_srgb8
        tr_ctx* c = g->members[k];
        TR_TRY(set_device(c));
        const size_t off = (size_t)c->band_y0 * c->width * 4, bytes = (size_t)(c->band_y1 - c->band_y0) * c->width * 4;
        TR_CUDA(cudaMemcpyAsync(rgba8 + off, c->srgb8.as<uint8_t>() + off, bytes, cudaMemcpyDeviceToHost, c->stream));
    }
    for (int k = 0; k < g->n; k++) {
        tr_ctx* c = g->members[k];
        TR_TRY(set_device(c));
        TR_CUDA(cudaStreamSynchronize(c->stream));
        TR_TRY(check_device_status(c, "tr_group_read_srgb8"));
    }
    return TR_OK;
}

}  // extern "C"
