// The routed calls of a hash-sharded index, one shard per handle (route -> all-to-all -> probe -> all-to-all -> place,
// include/classeq_b200.h), and the device buffers other processes can map for that exchange (CUDA IPC).
#include "capi_internal.hpp"

using namespace cls;

static int refuse_sharded(const cls_index *ix) {
    if (ix->shards.empty()) return CLS_OK;
    return fail(CLS_ERR_INVALID_ARGUMENT, "a sharded handle routes internally: the routed calls take the handle of one shard");
}

extern "C" {

int cls_routed_windows(cls_index *ix, cls_resident_batch *rb, uint64_t *n_windows) try {
    if (!ix || !rb || !n_windows) return fail(CLS_ERR_INVALID_ARGUMENT, "NULL argument");
    if (const int rc = refuse_sharded(ix)) return rc;
    CU_TRY(cudaSetDevice(ix->device));
    if (!rb->d_runs.p) {
        const PackedLayout &lay = rb->lay;
        const uint32_t k = ix->dix.k_size;
        uint64_t acc = 0;
        for (uint32_t j = 0; j < lay.n_device; ++j) acc += 2ull * (lay.lens[lay.perm[j]] - k + 1);
        CU_TRY(rb->d_route_state.reserve(256));
        CU_TRY(rb->d_runs.reserve((size_t)lay.n_device * 8 * sizeof(uint2) + 64));
        rb->n_windows = acc;
    }
    *n_windows = rb->n_windows;
    return CLS_OK;
} CLS_ABI_CATCH

static int route_hashes_impl(cls_index *ix, cls_resident_batch *rb, uint32_t n_shards, uint64_t seg_cap, uint64_t *const *seg_ptrs,
                             void *d_slot_win, uint64_t *counts_out, void *stream) {
    if ((uint64_t)n_shards * seg_cap >= 0xFFFFFFFFull) return fail(CLS_ERR_UNSUPPORTED, "send buffer beyond 2^32 entries: split the batch");
    uint64_t nw = 0;
    int rc = cls_routed_windows(ix, rb, &nw);
    if (rc != CLS_OK) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    unsigned long long *cursor = (unsigned long long *)rb->d_route_state.p;
    uint32_t *overflow = (uint32_t *)((char *)rb->d_route_state.p + 64);
    CU_TRY(cudaMemsetAsync(rb->d_route_state.p, 0, 128, st));
    for (const LengthClass &c : rb->lay.classes) {
        PlaceGeom g = make_place_geom(c.max_len, ix->dix.k_size, ix->dix.max_fanout);
        cudaError_t e = launch_route(ix->dix.k_size, (const uint32_t *)rb->d_words.p, (const ReadDesc *)rb->d_descs.p, c.first, c.count, g,
                                     n_shards, seg_cap, seg_ptrs, (uint16_t *)d_slot_win,
                                     (uint2 *)rb->d_runs.p, cursor, overflow, ix->sm_count, st);
        if (e == cudaErrorInvalidConfiguration)
            return fail(CLS_ERR_UNSUPPORTED, "the routed path places reads of up to 161 bases (the one-warp-per-read geometry)");
        if (e != cudaSuccess) return fail(CLS_ERR_CUDA, std::string("route kernel launch: ") + cudaGetErrorString(e));
    }
    uint64_t state[16];
    CU_TRY(cudaMemcpyAsync(state, rb->d_route_state.p, 128, cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaStreamSynchronize(st));
    if ((uint32_t)state[8]) return fail(CLS_ERR_OUT_OF_MEMORY, "a shard's segment of the send buffer is too small (seg_cap)");
    for (uint32_t o = 0; o < n_shards; ++o) counts_out[o] = state[o];
    return CLS_OK;
}

int cls_route_hashes(cls_index *ix, cls_resident_batch *rb, uint32_t n_shards, uint64_t seg_cap, void *d_send,
                     void *d_slot_win, uint64_t *counts_out, void *stream) try {
    if (!ix || !rb || !d_send || !d_slot_win || !counts_out) return fail(CLS_ERR_INVALID_ARGUMENT, "NULL argument");
    if (const int rc = refuse_sharded(ix)) return rc;
    if (n_shards == 0 || n_shards > kMaxShards) return fail(CLS_ERR_INVALID_ARGUMENT, "need 1 <= n_shards <= 8");
    uint64_t *seg[kMaxShards] = {nullptr};
    for (uint32_t o = 0; o < n_shards; ++o) seg[o] = (uint64_t *)d_send + (uint64_t)o * seg_cap;
    return route_hashes_impl(ix, rb, n_shards, seg_cap, seg, d_slot_win, counts_out, stream);
} CLS_ABI_CATCH

int cls_route_hashes_p2p(cls_index *ix, cls_resident_batch *rb, uint32_t n_shards, uint64_t seg_cap, void *const *d_segments,
                         void *d_slot_win, uint64_t *counts_out, void *stream) try {
    if (!ix || !rb || !d_segments || !d_slot_win || !counts_out) return fail(CLS_ERR_INVALID_ARGUMENT, "NULL argument");
    if (const int rc = refuse_sharded(ix)) return rc;
    if (n_shards == 0 || n_shards > kMaxShards) return fail(CLS_ERR_INVALID_ARGUMENT, "need 1 <= n_shards <= 8");
    uint64_t *seg[kMaxShards] = {nullptr};
    for (uint32_t o = 0; o < n_shards; ++o) {
        if (!d_segments[o]) return fail(CLS_ERR_INVALID_ARGUMENT, "NULL segment pointer");
        seg[o] = (uint64_t *)d_segments[o];
    }
    return route_hashes_impl(ix, rb, n_shards, seg_cap, seg, d_slot_win, counts_out, stream);
} CLS_ABI_CATCH

// ---- buffers other processes of the box can map (CUDA IPC): the inbox / reply box of the fused exchange ----
int cls_peer_alloc(int device, uint64_t bytes, void **d_ptr, uint8_t ipc_handle[64]) try {
    if (!d_ptr || !ipc_handle || bytes == 0) return fail(CLS_ERR_INVALID_ARGUMENT, "NULL argument or zero size");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
    CU_TRY(cudaSetDevice(device));
    void *p = nullptr;
    if (cudaMalloc(&p, bytes) != cudaSuccess) { cudaGetLastError(); return fail(CLS_ERR_OUT_OF_MEMORY, "cudaMalloc of a peer buffer failed"); }
    cudaIpcMemHandle_t h;
    cudaError_t e = cudaIpcGetMemHandle(&h, p);
    if (e != cudaSuccess) { cudaFree(p); return fail(CLS_ERR_CUDA, std::string("cudaIpcGetMemHandle: ") + cudaGetErrorString(e)); }
    std::memcpy(ipc_handle, &h, 64);
    *d_ptr = p;
    return CLS_OK;
} CLS_ABI_CATCH

int cls_peer_open(int device, const uint8_t ipc_handle[64], void **d_ptr) try {
    if (!d_ptr || !ipc_handle) return fail(CLS_ERR_INVALID_ARGUMENT, "NULL argument");
    CU_TRY(cudaSetDevice(device));
    cudaIpcMemHandle_t h;
    std::memcpy(&h, ipc_handle, 64);
    void *p = nullptr;
    cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) return fail(CLS_ERR_CUDA, std::string("cudaIpcOpenMemHandle: ") + cudaGetErrorString(e));
    *d_ptr = p;
    return CLS_OK;
} CLS_ABI_CATCH

int cls_peer_close(int device, void *d_ptr) try {
    if (!d_ptr) return CLS_OK;
    CU_TRY(cudaSetDevice(device));
    CU_TRY(cudaIpcCloseMemHandle(d_ptr));
    return CLS_OK;
} CLS_ABI_CATCH

int cls_peer_free(int device, void *d_ptr) try {
    if (!d_ptr) return CLS_OK;
    CU_TRY(cudaSetDevice(device));
    CU_TRY(cudaFree(d_ptr));
    return CLS_OK;
} CLS_ABI_CATCH

int cls_shard_probe(cls_index *ix, const void *d_hashes, uint64_t n, void *d_replies, void *stream) try {
    if (!ix || (n && (!d_hashes || !d_replies))) return fail(CLS_ERR_INVALID_ARGUMENT, "NULL argument");
    if (const int rc = refuse_sharded(ix)) return rc;
    CU_TRY(cudaSetDevice(ix->device));
    cudaError_t e = launch_shard_probe(ix->dix, ix->shard, (const uint64_t *)d_hashes, n, d_replies, (cudaStream_t)stream);
    if (e != cudaSuccess) return fail(CLS_ERR_CUDA, std::string("probe kernel launch: ") + cudaGetErrorString(e));
    return CLS_OK;
} CLS_ABI_CATCH

int cls_place_routed(cls_index *ix, cls_resident_batch *rb, const void *d_replies, const void *d_slot_win,
                     uint32_t n_shards, uint64_t seg_cap, const cls_params *params, void *stream) try {
    if (!ix || !rb || !params || !d_replies || !d_slot_win) return fail(CLS_ERR_INVALID_ARGUMENT, "NULL argument");
    if (const int rc = refuse_sharded(ix)) return rc;
    if (n_shards == 0 || n_shards > kMaxShards) return fail(CLS_ERR_INVALID_ARGUMENT, "need 1 <= n_shards <= 8");
    if (!rb->d_runs.p) return fail(CLS_ERR_INVALID_ARGUMENT, "cls_route_hashes has not run on this batch");
    CU_TRY(cudaSetDevice(ix->device));
    const PlaceParams pp = make_place_params(params);
    const int rc = grow_scratch(rb->d_scratch, (cudaStream_t)stream, scratch_for(rb->lay.classes, ix));
    if (rc != CLS_OK) return rc;
    for (const LengthClass &c : rb->lay.classes) {
        PlaceGeom g = make_place_geom(c.max_len, ix->dix.k_size, ix->dix.max_fanout);
        cudaError_t e = launch_place_routed(ix->dix, pp, (const uint32_t *)rb->d_words.p, (const ReadDesc *)rb->d_descs.p, c.first, c.count,
                                            (ResultRec *)rb->d_results.p, g, n_shards, seg_cap, (const uint2 *)rb->d_runs.p,
                                            (const uint16_t *)d_slot_win, d_replies, ix->sm_count, (cudaStream_t)stream,
                                            rb->d_scratch.p, rb->d_scratch.cap);
        if (e == cudaErrorInvalidConfiguration)
            return fail(CLS_ERR_UNSUPPORTED, "the routed path places reads of up to 161 bases (the one-warp-per-read geometry)");
        if (e != cudaSuccess) return fail(CLS_ERR_CUDA, std::string("routed place kernel launch: ") + cudaGetErrorString(e));
    }
    return CLS_OK;
} CLS_ABI_CATCH

}  // extern "C"
