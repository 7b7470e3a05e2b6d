// Host-side internals of the C ABI (include/classeq_b200.h) that its translation units share: capi.cpp (errors, index
// handles, debug exports), place_batch.cpp (planning, packing, cls_place_batch), resident.cpp (resident batches, text
// ingests), routed.cpp, capi_sharded.cpp and fastq_ingest.cpp.  Host code only: kernels are behind the *kernels.hpp.
#pragma once
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <mutex>
#include <new>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "../../include/classeq_b200.h"
#include "device_types.hpp"
#include "host_pool.hpp"
#include "index_build.hpp"
#include "kernels.hpp"
#include "last_error.hpp"

namespace cls {

inline int fail(int code, const std::string &msg) { return set_last_error(code, msg); }

// Nothing is thrown across the C ABI (include/classeq_b200.h, "Conventions"): every entry point with a body that
// can allocate is a function-try-block ending in CLS_ABI_CATCH.
int translate_exception();
#define CLS_ABI_CATCH catch (...) { return cls::translate_exception(); }

#define CU_TRY(expr)                                                                          \
    do {                                                                                      \
        cudaError_t _e = (expr);                                                              \
        if (_e != cudaSuccess)                                                                \
            return cls::fail(CLS_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e)); \
    } while (0)

inline double now_ms() {
    using namespace std::chrono;
    return duration<double, std::milli>(steady_clock::now().time_since_epoch()).count();
}

// ---- device / pinned buffers that grow on demand and are freed by their destructor ----------------------------------
// Growing frees the old block before the new one is allocated: nothing enqueued may still use it.  A buffer is freed
// with whatever device is current, so its owner makes its own device current before its buffers go.
template <cudaError_t (*Alloc)(void **, size_t), cudaError_t (*Free)(void *)>
struct Buf {
    void *p = nullptr;
    size_t cap = 0;
    Buf() = default;
    Buf(Buf &&o) noexcept : p(std::exchange(o.p, nullptr)), cap(std::exchange(o.cap, 0)) {}
    Buf &operator=(Buf &&o) noexcept { std::swap(p, o.p); std::swap(cap, o.cap); return *this; }
    ~Buf() { if (p) Free(p); }
    cudaError_t reserve(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) Free(p);
        p = nullptr; cap = 0;
        size_t want = bytes + bytes / 8 + 256;
        cudaError_t e = Alloc(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    template <class T> T *as() const { return static_cast<T *>(p); }
};
inline cudaError_t pin_alloc(void **p, size_t n) { return cudaHostAlloc(p, n, cudaHostAllocDefault); }
using DevBuf = Buf<cudaMalloc, cudaFree>;
using PinBuf = Buf<pin_alloc, cudaFreeHost>;

// One launch per length class: reads [first, first+count) of the length-ordered batch.
struct LengthClass {
    uint32_t first, count, max_len;
};

// Host-side view of a packed batch (buffers are owned by a Workspace, a ShardLane or a resident batch).
struct PackedLayout {
    uint64_t n_queries = 0;      // caller's batch size
    uint32_t n_device = 0;       // queries that reach the device (valid, L >= k)
    uint64_t n_words = 0;        // 32-bit words of packed bases
    std::vector<uint32_t> perm;  // device order -> caller index
    std::vector<uint8_t> pre_status;  // caller index -> status decided on the host, or 0xFF
    std::vector<uint32_t> lens;       // caller index -> query length (for n_query_kmers)
    std::vector<uint8_t> cls_id;      // caller index -> length class (scratch of plan_batch)
    std::vector<uint32_t> word_off;   // device order -> first packed word (+ one past the end)
    std::vector<LengthClass> classes;
};

// The buffers of one batch on its way through the device: packed bases, read descriptors and result records on both
// sides; the scan -> descent hand-over (every kernel of the batch runs on one stream: stream order protects its reuse);
// for packing on the device (pack_kernels.cu) the batch's ASCII bases, where every read starts in them and the
// invalid-base flags.
struct BatchBuffers {
    DevBuf d_words, d_descs, d_results, d_scratch, d_ascii, d_src, d_bad;
    PinBuf h_words, h_descs, h_results, h_src, h_bad;
};

// What one cls_place_batch call on a single-device handle works in (the handle's pool; reused across calls).
struct Workspace : BatchBuffers {
    cudaStream_t stream = nullptr, stream2 = nullptr, stream3 = nullptr;   // kernels; copies in; copies out
    std::vector<cudaEvent_t> chunk_ev;  // 4 per chunk: start, kernel start, kernel end, done
    PinBuf h_stage[2];                  // pinned staging ring for bases in pageable caller memory
    cudaEvent_t stage_ev[2] = {nullptr, nullptr};
    PackedLayout lay;                   // reused across calls
    bool in_use = false;
    ~Workspace() {   // (the handle's device is current) the streams are drained before the buffers go
        for (cudaStream_t s : {stream, stream2, stream3})
            if (s) { cudaStreamSynchronize(s); cudaStreamDestroy(s); }
        for (cudaEvent_t e : chunk_ev) if (e) cudaEventDestroy(e);
        for (cudaEvent_t e : stage_ev) if (e) cudaEventDestroy(e);
    }
};

// One shard of a sharded handle (cls_index_create_sharded), in both of its roles in a sub-batch: HOME of a part of the
// batch (its reads are packed, routed and placed on this shard's device) and OWNER of a slice of the table (it probes
// the hashes every home sent it).  All buffers live on `device`, are allocated once and grow only when a larger
// sub-batch needs them.
struct ShardLane : BatchBuffers {
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t route_ev = nullptr, probe_ev = nullptr;   // this home's hashes are in the owners' inboxes / this owner's replies are home
    cudaEvent_t t_begin = nullptr, t_end = nullptr;       // device time of the sub-batch on this lane (cls_get_timing)
    // owner side: n_shards segments of seg_cap hashes, segment h written by home h's route kernel (a peer store)
    DevBuf inbox;
    // home side: n_shards segments of seg_cap replies, segment o written by owner o's probe kernel; the window behind every
    // slot; the run of every read in every owner's segment; the per-owner cursors (bytes 0..63) and the overflow flag (64)
    DevBuf reply, slot_win, runs, state;
    PinBuf h_state, h_ascii;
    PackedLayout lay;
    bool dev_pack = false;  // this home's reads of the current sub-batch were packed on the device
    ~ShardLane() {   // the stream is drained, then the buffers go, on the lane's device
        cudaSetDevice(device);
        if (stream) { cudaStreamSynchronize(stream); cudaStreamDestroy(stream); }
        for (cudaEvent_t e : {route_ev, probe_ev, t_begin, t_end}) if (e) cudaEventDestroy(e);
    }
};

constexpr uint32_t kFastMaxLen = 162;   // longest read of the just-in-time plan (plan_reads_fast)
enum PackMode { kPackOnHost = 1, kPackOnDevice = 2, kPackMixed = 3 };

}  // namespace cls

struct cls_index {
    int device = 0;
    int sm_count = 0;
    uint32_t shard = 0, n_shards = 1;  // hash-sharded index: this handle holds the table entries of one shard
    struct Tables { cls::DevBuf table, arena, terms, qnodes, qchild, qid, qinfo, lca; } tables;   // what `dix` points into
    cls::DeviceIndex dix{};
    cls_index_info info{};
    std::mutex mu;
    std::vector<std::unique_ptr<cls::Workspace>> pool;
    cls_timing timing{};
    // a multi-device handle (cls_index_create_devices): one full index per listed device; this front object
    // owns no device memory of its own, and every call that works on one device goes to replicas[0]
    std::vector<std::unique_ptr<cls_index>> replicas;
    // a sharded handle (cls_index_create_sharded): shard s of the table on shards[s], its exchange state in lanes[s]; the
    // calls on such a handle run one at a time (call_mu)
    std::vector<std::unique_ptr<cls_index>> shards;
    std::vector<std::unique_ptr<cls::ShardLane>> lanes;
    std::mutex call_mu;
    // The calls that take another path on such a handle (capi_sharded.cpp).  The other units reach them only through
    // these pointers, so they link without capi_sharded.cpp against a CUDA runtime that has no peer-access calls.
    struct ShardedCalls {
        int (*place_batch)(cls_index *, const cls_batch *, const cls_params *, cls_result *);
        int (*place_resident)(cls_index *, cls_resident_batch *, const cls_params *, cudaStream_t);
    };
    const ShardedCalls *sharded = nullptr;
    ~cls_index() {   // also runs when cls_index_create fails half-way: nothing is leaked
        lanes.clear();    // first: the lanes' streams may still run kernels that read the shards' tables
        cudaSetDevice(device);
        pool.clear();     // then the workspaces, each drained before its buffers go
        tables = {};      // then its own buffers, before the shards and replicas (members) make their devices current
    }
};

struct cls_resident_batch {
    int device = 0;
    cls::PackedLayout lay;
    cls::DevBuf d_words, d_descs, d_results;
    cls::DevBuf d_scratch;  // scan -> descent hand-over (one placement of this batch in flight at a time)
    cls::DevBuf d_route_state, d_runs;  // routed path: per-owner cursors + overflow flag; the run of every read in every owner's segment
    std::vector<uint64_t> fa_header_begin, fa_header_end;  // cls_fasta_upload: the records the reader sent
    std::vector<uint32_t> fa_length;
    uint64_t n_windows = 0;
    cls::PinBuf h_results;
    ~cls_resident_batch() { cudaSetDevice(device); }   // its buffers are freed on its device (also on the upload calls' error paths)
};

namespace cls {

// ---- capi.cpp -------------------------------------------------------------------------------------------------------
int build_index_host(const cls_model_view *model, uint32_t shard, uint32_t n_shards, HostIndex &h);
int upload_index(const HostIndex &h, int device, uint32_t shard, uint32_t n_shards, std::unique_ptr<cls_index> &res);
PackMode resolve_pack_mode(size_t n_devices_of_handle, bool fast_plan, double &host_share);
bool is_pinned_host(const void *p);

// ---- place_batch.cpp ------------------------------------------------------------------------------------------------
int plan_batch(const cls_batch *batch, uint32_t k, uint32_t max_fanout, PackedLayout &lay, std::vector<uint32_t> &word_off);
bool plan_reads_fast(const cls_batch *batch, uint32_t k, PackedLayout &lay, std::vector<uint32_t> &word_off, uint64_t first,
                     uint64_t end, uint64_t &words_so_far, uint32_t &max_len, ReadDesc *descs, uint64_t *src, uint64_t base0);
void pack_batch(const cls_batch *batch, PackedLayout &lay, const std::vector<uint32_t> &word_off,
                uint32_t *words, ReadDesc *descs, uint64_t first = 0, uint64_t count = ~0ull);
uint64_t fill_pack_descs(const cls_batch *batch, const PackedLayout &lay, uint64_t base0, uint64_t first, uint64_t count,
                         ReadDesc *descs, uint64_t *src);
PlaceParams make_place_params(const cls_params *params);
size_t scratch_for(const std::vector<LengthClass> &classes, const cls_index *ix);
int grow_scratch(DevBuf &scratch, cudaStream_t stream, size_t bytes);
int launch_classes(cls_index *ix, const PackedLayout &lay, const cls_params *params, const uint32_t *d_words,
                   const ReadDesc *d_descs, ResultRec *d_results, cudaStream_t stream, DevBuf &scratch, uint64_t *launches);
void scatter_host_decided(const PackedLayout &lay, uint32_t k, cls_result *out, uint64_t first = 0, uint64_t end = ~0ull);
void scatter_device_range(const PackedLayout &lay, const ResultRec *recs, cls_result *out, uint64_t first, uint64_t count,
                          const uint8_t *bad = nullptr);
std::vector<uint64_t> cut_by_bases(const cls_batch *batch, size_t nd);
cls_result result_from(const cls_result *result, uint64_t a);

// ---- resident.cpp ---------------------------------------------------------------------------------------------------
// The handle a resident batch of `ix` lives on: a sharded handle's first shard, a multi-device handle's first device.
cls_index *resident_home(cls_index *ix);
// The end of a text ingest: the records (header slices, lengths, first kept base in the compacted codes) as a resident batch.
int ingest_finish(cls_index *home, const uint8_t *d_codes, std::vector<uint64_t> &hb, std::vector<uint64_t> &he, std::vector<uint32_t> &ln,
                  const std::vector<uint64_t> &src, cudaStream_t st, cls_resident_batch **out, cls_fasta_records *records);

// ---- one row of the caller's result arrays --------------------------------------------------------------------------
// Every field but status and n_query_kmers, of a query whose status was decided without a placement.
inline void zero_row(cls_result *out, uint64_t i) {
    if (out->node_id) out->node_id[i] = 0;
    if (out->one) out->one[i] = 0;
    if (out->rest) out->rest[i] = 0;
    if (out->n_matched) out->n_matched[i] = 0;
    if (out->n_root_matched) out->n_root_matched[i] = 0;
    if (out->iterations) out->iterations[i] = 0;
}
// Every field but n_query_kmers, from the device's result record.
inline void write_row(cls_result *out, uint64_t i, const ResultRec &r) {
    if (out->status) out->status[i] = (uint8_t)r.status;
    if (out->node_id) out->node_id[i] = r.node_id;
    if (out->one) out->one[i] = r.one;
    if (out->rest) out->rest[i] = r.rest;
    if (out->n_matched) out->n_matched[i] = r.n_matched;
    if (out->n_root_matched) out->n_root_matched[i] = r.n_root_matched;
    if (out->iterations) out->iterations[i] = r.iterations;
}

}  // namespace cls
