// C ABI of the placement path (include/classeq_b200.h).  Host-side plumbing only: 2-bit packing
// and length ordering of the batch, pinned staging, stream/event management, and the scatter of
// the 32-byte device result records into the caller's arrays.  All arithmetic of the path runs
// in kernels.cu; there is no CPU fallback anywhere in this file.
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <mutex>
#include <new>
#include <stdexcept>
#include <string>
#include <thread>
#include <vector>

#include "../../include/classeq_b200.h"
#include "device_types.hpp"
#include "index_build.hpp"
#include "host_pack.hpp"
#include "fasta_kernels.hpp"
#include "host_pool.hpp"
#include "kernels.hpp"
#include "murmur3_host.hpp"

using namespace cls;

namespace {

thread_local std::string g_last_error;

int fail(int code, const std::string &msg) {
    g_last_error = msg;
    return code;
}

}  // namespace
namespace cls {
int set_last_error(int code, const std::string &msg) { return fail(code, msg); }  // for host_api.cpp
}
namespace {

// Nothing is thrown across the C ABI (include/classeq_b200.h, "Conventions"): every entry point with a body that
// can allocate is a function-try-block ending in CLS_ABI_CATCH.
int translate_exception() {
    try {
        throw;
    } catch (const std::bad_alloc &) {
        return fail(CLS_ERR_OUT_OF_MEMORY, "host allocation failed");
    } catch (const std::exception &e) {
        return fail(CLS_ERR_INVALID_ARGUMENT, std::string("unexpected exception: ") + e.what());
    } catch (...) {
        return fail(CLS_ERR_INVALID_ARGUMENT, "unexpected exception");
    }
}
#define CLS_ABI_CATCH catch (...) { return translate_exception(); }

}  // namespace
namespace {

#define CU_TRY(expr)                                                                          \
    do {                                                                                      \
        cudaError_t _e = (expr);                                                              \
        if (_e != cudaSuccess)                                                                \
            return fail(CLS_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e));    \
    } while (0)

double now_ms() {
    using namespace std::chrono;
    return duration<double, std::milli>(steady_clock::now().time_since_epoch()).count();
}

// ---- device / pinned buffers that grow on demand --------------------------------------------
struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    cudaError_t reserve(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        size_t want = bytes + bytes / 8 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};
struct PinBuf {
    void *p = nullptr;
    size_t cap = 0;
    cudaError_t reserve(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFreeHost(p);
        p = nullptr; cap = 0;
        size_t want = bytes + bytes / 8 + 256;
        cudaError_t e = cudaHostAlloc(&p, want, cudaHostAllocDefault);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
};

// One launch per length class: reads [first, first+count) of the length-ordered batch.
struct LengthClass {
    uint32_t first, count, max_len;
};

// Host-side view of a packed batch (buffers are owned by a Workspace or a resident batch).
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

struct Workspace {
    cudaStream_t stream = nullptr, stream2 = nullptr, stream3 = nullptr;   // kernels; copies in; copies out
    std::vector<cudaEvent_t> chunk_ev;  // 4 per chunk: start, kernel start, kernel end, done
    PinBuf h_words, h_descs, h_results;
    DevBuf d_words, d_descs, d_results;
    DevBuf d_scratch;                   // scan -> descent hand-over (every kernel runs on `stream`: stream order protects its reuse)
    // packing on the device (pack_kernels.cu): the batch's ASCII bases, where every read starts in them, invalid-base flags
    DevBuf d_ascii, d_src, d_bad;
    PinBuf h_src, h_bad, h_stage[2];    // h_stage: pinned staging ring for bases in pageable caller memory
    cudaEvent_t stage_ev[2] = {nullptr, nullptr};
    PackedLayout lay;                   // reused across calls
    bool in_use = false;
};

// One shard of a sharded handle (cls_index_create_sharded), in both of its roles in a sub-batch: HOME of a part of the
// batch (its reads are packed, routed and placed on this shard's device) and OWNER of a slice of the table (it probes
// the hashes every home sent it).  All buffers live on `device`, are allocated once and grow only when a larger
// sub-batch needs them.
struct ShardLane {
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t route_ev = nullptr, probe_ev = nullptr;   // this home's hashes are in the owners' inboxes / this owner's replies are home
    cudaEvent_t t_begin = nullptr, t_end = nullptr;       // device time of the sub-batch on this lane (cls_get_timing)
    // owner side: n_shards segments of seg_cap hashes, segment h written by home h's route kernel (a peer store)
    DevBuf inbox;
    // home side: n_shards segments of seg_cap replies, segment o written by owner o's probe kernel; the window behind every
    // slot; the run of every read in every owner's segment; the per-owner cursors (bytes 0..63) and the overflow flag (64)
    DevBuf reply, slot_win, runs, state;
    DevBuf d_words, d_descs, d_results, d_scratch, d_ascii, d_src, d_bad;
    PinBuf h_words, h_descs, h_results, h_state, h_src, h_bad, h_ascii;
    PackedLayout lay;
    bool dev_pack = false;  // this home's reads of the current sub-batch were packed on the device
    ShardLane() = default;
    ShardLane(const ShardLane &) = delete;
    ShardLane &operator=(const ShardLane &) = delete;
    ~ShardLane() {
        cudaSetDevice(device);
        if (stream) { cudaStreamSynchronize(stream); cudaStreamDestroy(stream); }
        for (cudaEvent_t e : {route_ev, probe_ev, t_begin, t_end}) if (e) cudaEventDestroy(e);
        for (DevBuf *b : {&inbox, &reply, &slot_win, &runs, &state, &d_words, &d_descs, &d_results, &d_scratch, &d_ascii, &d_src, &d_bad})
            b->release();
        for (PinBuf *b : {&h_words, &h_descs, &h_results, &h_state, &h_src, &h_bad, &h_ascii}) b->release();
    }
};

}  // namespace

struct cls_index {
    int device = 0;
    int sm_count = 0;
    uint32_t shard = 0, n_shards = 1;  // hash-sharded index: this handle holds the table entries of one shard
    DevBuf d_table, d_arena, d_terms, d_qnodes, d_qchild, d_qid, d_qinfo, d_lca;
    DeviceIndex dix{};
    cls_index_info info{};
    std::mutex mu;
    std::vector<std::unique_ptr<Workspace>> pool;
    cls_timing timing{};
    // a multi-device handle (cls_index_create_devices): one full index per listed device; this front object
    // owns no device memory of its own, and every call that works on one device goes to replicas[0]
    std::vector<std::unique_ptr<cls_index>> replicas;
    // a sharded handle (cls_index_create_sharded): shard s of the table on shards[s], its exchange state in lanes[s]; the
    // calls on such a handle run one at a time (call_mu)
    std::vector<std::unique_ptr<cls_index>> shards;
    std::vector<std::unique_ptr<ShardLane>> lanes;
    std::mutex call_mu;
    struct ShardedCalls {   // the calls that take another path on such a handle (capi_sharded.cu)
        int (*place_batch)(cls_index *, const cls_batch *, const cls_params *, cls_result *);
        int (*place_resident)(cls_index *, cls_resident_batch *, const cls_params *, cudaStream_t);
    };
    const ShardedCalls *sharded = nullptr;
    cls_index() = default;
    cls_index(const cls_index &) = delete;
    cls_index &operator=(const cls_index &) = delete;
    ~cls_index() {   // also runs when cls_index_create fails half-way: nothing is leaked
        lanes.clear();   // (before the shards: the lanes' streams may still run kernels that read the shards' tables)
        cudaSetDevice(device);
        for (auto &w : pool) {
            for (cudaStream_t s : {w->stream, w->stream2, w->stream3}) { cudaStreamSynchronize(s); cudaStreamDestroy(s); }
            for (auto &e : w->chunk_ev) if (e) cudaEventDestroy(e);
            w->h_words.release(); w->h_descs.release(); w->h_results.release();
            w->d_words.release(); w->d_descs.release(); w->d_results.release();
            w->d_scratch.release();
            for (auto &e : w->stage_ev) if (e) cudaEventDestroy(e);
            w->d_ascii.release(); w->d_src.release(); w->d_bad.release();
            w->h_src.release(); w->h_bad.release(); w->h_stage[0].release(); w->h_stage[1].release();
        }
        d_table.release(); d_arena.release(); d_qnodes.release(); d_qchild.release(); d_qid.release();
        d_terms.release(); d_qinfo.release(); d_lca.release();
    }
};

struct cls_resident_batch {
    int device = 0;
    PackedLayout lay;
    DevBuf d_words, d_descs, d_results;
    DevBuf d_scratch;  // scan -> descent hand-over (one placement of this batch in flight at a time)
    DevBuf d_route_state, d_runs;  // routed path: per-owner cursors + overflow flag; the run of every read in every owner's segment
    std::vector<uint64_t> fa_header_begin, fa_header_end;  // cls_fasta_upload: the records the reader sent
    std::vector<uint32_t> fa_length;
    uint64_t n_windows = 0;
    PinBuf h_results;
    cls_resident_batch() = default;
    cls_resident_batch(const cls_resident_batch &) = delete;
    cls_resident_batch &operator=(const cls_resident_batch &) = delete;
    ~cls_resident_batch() {   // also runs on the error paths of the upload calls: nothing is leaked
        cudaSetDevice(device);
        d_words.release(); d_descs.release(); d_results.release(); d_scratch.release();
        d_route_state.release(); d_runs.release(); h_results.release();
    }
};

namespace {

// Decide host-side statuses, group the surviving queries into LENGTH CLASSES (all reads of a class
// share one per-read table geometry; longest class first so that long reads start first; input
// order is kept inside a class), and compute the packed layout.
int plan_batch(const cls_batch *batch, uint32_t k, uint32_t max_fanout, PackedLayout &lay,
               std::vector<uint32_t> &word_off) {
    const uint64_t n = batch->n_queries;
    if (n >= 0xFFFFFFFFull) return fail(CLS_ERR_INVALID_ARGUMENT, "more than 2^32-1 queries in one batch");
    if (n && (!batch->offsets || (batch->offsets[n] && !batch->bases)))
        return fail(CLS_ERR_INVALID_ARGUMENT, "batch arrays are NULL");
    lay.classes.clear();               // buffers are reused from call to call (no fresh pages)
    lay.n_queries = n;
    lay.n_device = 0;
    lay.n_words = 0;
    lay.pre_status.resize(n);
    lay.lens.resize(n);
    // class id = log2 of the de-duplication table size for that length (make_place_geom)
    constexpr int kMaxClass = 40;
    auto class_of = [k](uint64_t len) {
        const uint64_t h2 = 4 * (len - k + 1);
        int c = 6;
        while ((1ull << c) < h2) ++c;
        return c;
    };
    // Everything below runs over fixed blocks of reads on the host pool: per-block class histograms,
    // a short serial scan over (class, block), then every block fills its own slice of the permutation
    // (input order is kept inside a class, exactly as a serial pass would).
    constexpr uint64_t kBlock = 1 << 15;
    const uint64_t nblk = (n + kBlock - 1) / kBlock;
    std::vector<uint64_t> bcount(nblk * kMaxClass, 0), bwords(nblk * kMaxClass, 0), bmax(nblk * kMaxClass, 0);
    std::vector<uint8_t> &cls_id = lay.cls_id;
    cls_id.resize(n);
    std::atomic<bool> bad_offsets{false}, too_long{false};
    parallel_for(nblk, 1, [&](uint64_t b0, uint64_t b1) {  // per-read lengths, statuses, classes
        for (uint64_t blk = b0; blk < b1; ++blk) {
            uint64_t *bc = &bcount[blk * kMaxClass], *bw = &bwords[blk * kMaxClass], *bm = &bmax[blk * kMaxClass];
            const uint64_t hi = std::min(n, (blk + 1) * kBlock);
            for (uint64_t i = blk * kBlock; i < hi; ++i) {
                lay.pre_status[i] = 0xFF;
                cls_id[i] = 0xFF;
                if (batch->offsets[i] > batch->offsets[i + 1]) { bad_offsets = true; continue; }
                const uint64_t len = batch->offsets[i + 1] - batch->offsets[i];
                if (len >= (1ull << 31)) { too_long = true; continue; }
                lay.lens[i] = (uint32_t)len;
                if (len < k) { lay.pre_status[i] = CLS_STATUS_ERR_TOO_SHORT; continue; }  // kmers_map.rs:383-385
                const int c = class_of(len);
                cls_id[i] = (uint8_t)c;
                bc[c]++;
                bw[c] += (len + 15u) / 16u;
                bm[c] = std::max<uint64_t>(bm[c], len);
            }
        }
    });
    if (bad_offsets) return fail(CLS_ERR_INVALID_ARGUMENT, "batch offsets are not non-decreasing");
    if (too_long) return fail(CLS_ERR_INVALID_ARGUMENT, "query longer than 2^31 bases");
    uint64_t acc = 0, w = 0;
    for (int c = kMaxClass - 1; c >= 0; --c) {  // longest class first; bcount / bwords become the blocks' start positions
        uint64_t cnt = 0, mx = 0;
        const uint64_t first = acc;
        for (uint64_t blk = 0; blk < nblk; ++blk) {
            const uint64_t bc = bcount[blk * kMaxClass + c], bw = bwords[blk * kMaxClass + c];
            bcount[blk * kMaxClass + c] = acc; bwords[blk * kMaxClass + c] = w;
            acc += bc; w += bw; cnt += bc;
            mx = std::max(mx, bmax[blk * kMaxClass + c]);
        }
        if (cnt) lay.classes.push_back(LengthClass{(uint32_t)first, (uint32_t)cnt, (uint32_t)mx});
    }
    if (w >= 0xFFFFFFFFull) return fail(CLS_ERR_INVALID_ARGUMENT, "batch exceeds 2^32 packed words; split it");
    lay.n_device = (uint32_t)acc;
    lay.n_words = w;
    lay.perm.resize(acc);
    word_off.resize((size_t)acc + 1);
    parallel_for(nblk, 1, [&](uint64_t b0, uint64_t b1) {
        for (uint64_t blk = b0; blk < b1; ++blk) {
            uint64_t *start = &bcount[blk * kMaxClass], *wstart = &bwords[blk * kMaxClass];
            const uint64_t hi = std::min(n, (blk + 1) * kBlock);
            for (uint64_t i = blk * kBlock; i < hi; ++i) {
                const uint8_t c = cls_id[i];
                if (c == 0xFF) continue;
                const uint64_t j = start[c]++;
                lay.perm[j] = (uint32_t)i;
                word_off[j] = (uint32_t)wstart[c];
                wstart[c] += (lay.lens[i] + 15u) / 16u;
            }
        }
    });
    word_off[acc] = (uint32_t)w;
    (void)max_fanout;
    return CLS_OK;
}

// Pack the planned batch into `words`/`descs` (pinned).  Invalid bases demote the query to
// CLS_STATUS_ERR_INVALID_BASE; it still occupies its device slot (the device result is ignored).
void pack_batch(const cls_batch *batch, PackedLayout &lay, const std::vector<uint32_t> &word_off,
                uint32_t *words, ReadDesc *descs, uint64_t first = 0, uint64_t count = ~0ull) {
    if (count == ~0ull) count = lay.n_device;
    parallel_for(count, 4096, [&](uint64_t a0, uint64_t b0) {
        for (uint64_t j = first + a0; j < first + b0; ++j) {
            const uint64_t i = lay.perm[j];
            const uint32_t len = (uint32_t)(batch->offsets[i + 1] - batch->offsets[i]);
            descs[j] = ReadDesc{word_off[j], len};
            if (!pack_read(batch->bases + batch->offsets[i], len, words + word_off[j]))
                lay.pre_status[i] = CLS_STATUS_ERR_INVALID_BASE;
        }
    });
}

PlaceParams make_place_params(const cls_params *params) {
    PlaceParams pp;
    pp.max_iterations = params->max_iterations;
    pp.remove_intersection = params->remove_intersection ? 1u : 0u;
    double cov = params->min_match_coverage;  // place_sequence.rs:67-75
    if (std::isnan(cov)) cov = 0.0;           // NaN survives the clamp and `NaN as usize` is 0
    else if (cov > 1.0) cov = 1.0;
    else if (cov < 0.0) cov = 0.0;
    pp.min_match_coverage = cov;
    return pp;
}

int launch_classes(cls_index *ix, const PackedLayout &lay, const cls_params *params, const uint32_t *d_words,
                   const ReadDesc *d_descs, ResultRec *d_results, cudaStream_t stream, DevBuf &scratch, uint64_t *launches) {
    const PlaceParams pp = make_place_params(params);
    size_t want = 0;
    for (const LengthClass &c : lay.classes) {
        want = std::max(want, place_scratch_bytes(c.count, c.max_len, ix->dix.k_size, ix->dix.max_fanout));
    }
    if (want > scratch.cap) {
        if (scratch.p) CU_TRY(cudaStreamSynchronize(stream));  // an earlier placement on this stream may still use it
        CU_TRY(scratch.reserve(want));
    }
    for (const LengthClass &c : lay.classes) {
        PlaceGeom g = make_place_geom(c.max_len, ix->dix.k_size, ix->dix.max_fanout);
        uint32_t nl = 0;
        cudaError_t e = launch_place(ix->dix, pp, d_words, d_descs, c.first, c.count, d_results, g, ix->sm_count, stream,
                                     scratch.p, scratch.cap, &nl);
        if (launches) *launches += nl;
        if (e == cudaErrorInvalidConfiguration)
            return fail(CLS_ERR_UNSUPPORTED, "query too long (or tree fan-out too large) for the per-warp shared-memory tables");
        if (e != cudaSuccess) return fail(CLS_ERR_CUDA, std::string("place kernel launch: ") + cudaGetErrorString(e));
    }
    return CLS_OK;
}

// Fields decided on the host (n_query_kmers of every query; everything for queries that never
// reach the device).
// (queries [first, end) in caller order: cls_place_batch writes them piece by piece between its chunks)
void scatter_host_decided(const PackedLayout &lay, uint32_t k, cls_result *out, uint64_t first = 0, uint64_t end = ~0ull) {
    if (end > lay.n_queries) end = lay.n_queries;
    if (first >= end) return;
    parallel_for(end - first, 65536, [&](uint64_t a0, uint64_t b0) {
        for (uint64_t i = first + a0; i < first + b0; ++i) {
            const uint64_t len = lay.lens[i];
            const uint8_t ps = lay.pre_status[i];
            if (out->n_query_kmers) out->n_query_kmers[i] = len >= k ? (uint32_t)(2 * (len - k + 1)) : 0u;
            if (ps != 0xFF) {
                if (out->status) out->status[i] = ps;
                if (out->node_id) out->node_id[i] = 0;
                if (out->one) out->one[i] = 0;
                if (out->rest) out->rest[i] = 0;
                if (out->n_matched) out->n_matched[i] = 0;
                if (out->n_root_matched) out->n_root_matched[i] = 0;
                if (out->iterations) out->iterations[i] = 0;
            }
        }
    });
}

// Device result records [first, first + count) (device order) -> the caller's arrays (caller order).
// Queries demoted on the host while packing (invalid base) keep their host status.
void scatter_device_range(const PackedLayout &lay, const ResultRec *recs, cls_result *out, uint64_t first, uint64_t count,
                          const uint8_t *bad = nullptr) {
    parallel_for(count, 65536, [&](uint64_t a, uint64_t b) {
        for (uint64_t j = first + a; j < first + b; ++j) {
            const uint64_t i = lay.perm[j];
            const ResultRec &r = recs[j];
            if (lay.pre_status[i] != 0xFF || (bad && bad[j])) {   // bad: flagged by the device packer
                if (out->status) out->status[i] = lay.pre_status[i] != 0xFF ? lay.pre_status[i] : (uint8_t)CLS_STATUS_ERR_INVALID_BASE;
                if (out->node_id) out->node_id[i] = 0;
                if (out->one) out->one[i] = 0;
                if (out->rest) out->rest[i] = 0;
                if (out->n_matched) out->n_matched[i] = 0;
                if (out->n_root_matched) out->n_root_matched[i] = 0;
                if (out->iterations) out->iterations[i] = 0;
                continue;
            }
            if (out->status) out->status[i] = (uint8_t)r.status;
            if (out->node_id) out->node_id[i] = r.node_id;
            if (out->one) out->one[i] = r.one;
            if (out->rest) out->rest[i] = r.rest;
            if (out->n_matched) out->n_matched[i] = r.n_matched;
            if (out->n_root_matched) out->n_root_matched[i] = r.n_root_matched;
            if (out->iterations) out->iterations[i] = r.iterations;
        }
    });
}

void scatter_results(const PackedLayout &lay, uint32_t k, const ResultRec *recs, cls_result *out) {
    scatter_host_decided(lay, k, out);
    scatter_device_range(lay, recs, out, 0, lay.n_device);
}

Workspace *acquire_ws(cls_index *ix) {
    std::lock_guard<std::mutex> lk(ix->mu);
    for (auto &w : ix->pool)
        if (!w->in_use) { w->in_use = true; return w.get(); }
    auto w = std::make_unique<Workspace>();
    bool ok = true;
    for (cudaStream_t *s : {&w->stream, &w->stream2, &w->stream3})
        if (ok) ok = cudaStreamCreateWithFlags(s, cudaStreamNonBlocking) == cudaSuccess;
    if (!ok) {   // nothing half-made is left behind
        for (cudaStream_t s : {w->stream, w->stream2, w->stream3}) if (s) cudaStreamDestroy(s);
        return nullptr;
    }
    w->in_use = true;
    ix->pool.push_back(std::move(w));
    return ix->pool.back().get();
}

void release_ws(cls_index *ix, Workspace *w) {
    std::lock_guard<std::mutex> lk(ix->mu);
    w->in_use = false;
}

// Returns the workspace to the pool when the call ends.  If the call leaves before it has drained its own work
// (`clean` still false: an error path after the first enqueue), copies and kernels may still be in flight on the
// workspace's streams, using its pinned and device buffers: they are waited for first, so that the next caller that
// takes the workspace cannot overwrite (or re-reserve, i.e. free) buffers the GPU is still working on.
struct WsGuard {
    cls_index *ix;
    Workspace *w;
    bool clean = false;
    ~WsGuard() {
        if (!w) return;
        if (!clean)
            for (cudaStream_t s : {w->stream, w->stream2, w->stream3}) cudaStreamSynchronize(s);
        release_ws(ix, w);
    }
};

}  // namespace

extern "C" {

int cls_abi_version(void) { return CLS_ABI_VERSION; }

const char *cls_last_error(void) { return g_last_error.c_str(); }

void cls_params_default(cls_params *p) {
    if (!p) return;
    p->max_iterations = 1000;      // place_sequence.rs:65
    p->remove_intersection = 0;    // place_sequence.rs:64
    p->min_match_coverage = 0.7;   // place_sequence.rs:74
}

int cls_device_count(void) try {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) return fail(CLS_ERR_CUDA, std::string("cudaGetDeviceCount: ") + cudaGetErrorString(e));
    return n;
} CLS_ABI_CATCH

int cls_index_create(const cls_model_view *model, int device, cls_index **out) try {
    return cls_index_create_shard(model, device, 0, 1, out);
} CLS_ABI_CATCH

// The host-built index `h` on one device.
static int upload_index(const HostIndex &h, int device, uint32_t shard, uint32_t n_shards, std::unique_ptr<cls_index> &res) {
    CU_TRY(cudaSetDevice(device));
    cudaDeviceProp prop;
    CU_TRY(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) return fail(CLS_ERR_CUDA, "this library only carries sm_100a code; device is sm_" + std::to_string(prop.major) + std::to_string(prop.minor));
    auto ix = std::make_unique<cls_index>();
    ix->device = device;
    ix->sm_count = prop.multiProcessorCount;
    ix->shard = shard;
    ix->n_shards = n_shards;
    auto up = [&](DevBuf &b, const void *src, size_t bytes) -> cudaError_t {
        cudaError_t e = b.reserve(std::max<size_t>(bytes, 16));
        if (e != cudaSuccess) return e;
        return bytes ? cudaMemcpy(b.p, src, bytes, cudaMemcpyHostToDevice) : cudaSuccess;
    };
    CU_TRY(up(ix->d_table, h.table.data(), h.table.size() * sizeof(Slot)));
    CU_TRY(up(ix->d_arena, h.arena.data(), h.arena.size() * sizeof(SetWord)));
    CU_TRY(up(ix->d_qnodes, h.qnodes.data(), h.qnodes.size() * sizeof(QNode)));
    CU_TRY(up(ix->d_qchild, h.q_child_list.data(), h.q_child_list.size() * sizeof(uint32_t)));
    CU_TRY(up(ix->d_qid, h.q_node_id.data(), h.q_node_id.size() * sizeof(uint64_t)));
    CU_TRY(up(ix->d_terms, h.terms.data(), h.terms.size() * sizeof(uint32_t)));
    CU_TRY(up(ix->d_qinfo, h.qinfo.data(), h.qinfo.size() * sizeof(QInfo)));
    CU_TRY(up(ix->d_lca, h.lca_table.data(), h.lca_table.size() * sizeof(uint64_t)));
    ix->dix.table = (const Slot *)ix->d_table.p;
    ix->dix.bucket_mask = h.n_buckets - 1;
    ix->dix.arena = (const SetWord *)ix->d_arena.p;
    ix->dix.qnodes = (const QNode *)ix->d_qnodes.p;
    ix->dix.q_child_list = (const uint32_t *)ix->d_qchild.p;
    ix->dix.q_node_id = (const uint64_t *)ix->d_qid.p;
    ix->dix.terms = (const uint32_t *)ix->d_terms.p;
    ix->dix.qinfo = (const QInfo *)ix->d_qinfo.p;
    ix->dix.lca_table = (const uint64_t *)ix->d_lca.p;
    ix->dix.n_q = (uint32_t)h.qnodes.size();
    ix->dix.euler_len = h.euler_len;
    ix->dix.closed = h.closed ? 1u : 0u;
    ix->dix.k_size = h.k_size;
    ix->dix.m_eff = h.m_eff;
    ix->dix.max_fanout = h.max_fanout;
    ix->dix.root_children_none = h.root_children_none ? 1u : 0u;
    ix->info.k_size = h.k_size;
    ix->info.m_size = h.m_size;
    ix->info.n_entries = h.n_entries_kept;
    ix->info.n_buckets = h.n_buckets;
    ix->info.table_bytes = h.table.size() * sizeof(Slot);
    ix->info.n_distinct_sets = h.n_distinct_sets;
    ix->info.set_arena_bytes = h.closed ? h.terms.size() * sizeof(uint32_t) : h.arena.size() * sizeof(SetWord);
    ix->info.closed_sets = h.closed ? 1u : 0u;
    ix->info.n_nonleaf_nodes = h.qnodes.size();
    ix->info.max_nonleaf_fanout = h.max_fanout;
    ix->info.device = device;
    ix->info.n_devices = 1;
    res = std::move(ix);
    return CLS_OK;
}

static int build_index_host(const cls_model_view *model, uint32_t shard, uint32_t n_shards, HostIndex &h) {
    std::string err;
    int rc = build_host_index(model, h, err, shard, n_shards);
    if (rc != CLS_OK) return fail(rc, err);
    if (h.n_buckets > (1ull << (n_shards > 1 ? 28 : 30))) return fail(CLS_ERR_UNSUPPORTED, "k-mer table too large (2^30 buckets, 2^28 per shard)");
    return CLS_OK;
}

int cls_index_create_shard(const cls_model_view *model, int device, uint32_t shard, uint32_t n_shards, cls_index **out) try {
    if (!out) return fail(CLS_ERR_INVALID_ARGUMENT, "out is NULL");
    *out = nullptr;
    if (n_shards == 0 || n_shards > kMaxShards || shard >= n_shards)
        return fail(CLS_ERR_INVALID_ARGUMENT, "need 1 <= n_shards <= 8 and shard < n_shards");
    HostIndex h;
    int rc = build_index_host(model, shard, n_shards, h);
    if (rc != CLS_OK) return rc;
    std::unique_ptr<cls_index> ix;
    if ((rc = upload_index(h, device, shard, n_shards, ix)) != CLS_OK) return rc;
    *out = ix.release();
    return CLS_OK;
} CLS_ABI_CATCH

int cls_index_create_devices(const cls_model_view *model, uint32_t n_devices, const int *devices, cls_index **out) try {
    if (!out) return fail(CLS_ERR_INVALID_ARGUMENT, "out is NULL");
    *out = nullptr;
    if (n_devices == 0 || n_devices > 64 || !devices) return fail(CLS_ERR_INVALID_ARGUMENT, "need 1 <= n_devices <= 64 and a device list");
    HostIndex h;
    int rc = build_index_host(model, 0, 1, h);   // built once, uploaded to every device
    if (rc != CLS_OK) return rc;
    auto front = std::make_unique<cls_index>();
    for (uint32_t d = 0; d < n_devices; ++d) {
        std::unique_ptr<cls_index> rep;
        if ((rc = upload_index(h, devices[d], 0, 1, rep)) != CLS_OK) return rc;
        front->replicas.push_back(std::move(rep));
    }
    front->device = front->replicas[0]->device;
    front->sm_count = front->replicas[0]->sm_count;
    front->dix = front->replicas[0]->dix;
    front->info = front->replicas[0]->info;
    front->info.n_devices = n_devices;
    *out = front.release();
    return CLS_OK;
} CLS_ABI_CATCH

int cls_index_create_multi(const cls_model_view *model, uint64_t device_mask, cls_index **out) try {
    if (!out) return fail(CLS_ERR_INVALID_ARGUMENT, "out is NULL");
    *out = nullptr;
    int n = 0;
    CU_TRY(cudaGetDeviceCount(&n));
    std::vector<int> devs;
    for (int d = 0; d < n && d < 64; ++d)
        if (device_mask == 0 || ((device_mask >> d) & 1ull)) devs.push_back(d);
    if (devs.empty()) return fail(CLS_ERR_INVALID_ARGUMENT, "device_mask names no visible CUDA device");
    if (device_mask >> (n < 64 ? n : 63) > (n < 64 ? 0ull : 1ull)) return fail(CLS_ERR_INVALID_ARGUMENT, "device_mask names a device that is not visible");
    return cls_index_create_devices(model, (uint32_t)devs.size(), devs.data(), out);
} CLS_ABI_CATCH

void cls_index_destroy(cls_index *ix) { delete ix; }

int cls_index_get_info(const cls_index *ix, cls_index_info *info) try {
    if (!ix || !info) return fail(CLS_ERR_INVALID_ARGUMENT, "NULL argument");
    *info = ix->info;
    return CLS_OK;
} CLS_ABI_CATCH

// Where the 2-bit packing of a cls_place_batch call runs.  On the host (AVX-512 / AVX2 packer on the host pool, 38 bytes
// per 150-base read cross PCIe) when the process has cores to spare; on the device (the ASCII bases cross PCIe as they
// are, 150 bytes per read - straight from the caller's memory when it is pinned, else through a pinned staging ring -
// and pack_kernels.cu packs them) when several GPUs share few host cores: eight ranks of a 32-core box each packed
// with their share of the cores and the 1 -> 8 GPU end-to-end curve collapsed (SCALE_r01: efficiency 0.33).
// CLS_PACK=host|device forces the choice; the default is "device" below sixteen cores per GPU in use (two GPUs on a 24-core box: 31.2 against 35.7 ms per 5 M reads, profiles/r2b).
// Mixed (cls_set_pack_mode(3), CLS_PACK=mixed; batches of short reads only): the chunks of a call are dealt to both - the
// host cores pack some while the copy engine moves the ASCII of the others - in the ratio that would let the two finish
// together (about 2.5 GB/s of ASCII per core against about 24 GB/s per GPU).  Never the automatic choice: on the
// boxes measured it lost to device packing (8 GPUs, 32 cores: 23.5 against 20.4 ms per step - the host cores are the
// scarcer resource there, and the 20 ms are the 1.66 GB of a step crossing PCIe at the 83 GB/s the eight GPUs get
// together; profiles/r2b/bench_cfg3_n8_*.json).
static std::atomic<int> g_pack_mode{-1};   // cls_set_pack_mode; -1: not set, CLS_PACK decides
enum PackMode { kPackOnHost = 1, kPackOnDevice = 2, kPackMixed = 3 };
static PackMode resolve_pack_mode(size_t n_devices_of_handle, bool fast_plan, double &host_share) {
    static const int env = [] {
        const char *e = getenv("CLS_PACK");
        if (!e) return 0;
        return !strcmp(e, "device") ? 2 : !strcmp(e, "host") ? 1 : !strcmp(e, "mixed") ? 3 : 0;
    }();
    unsigned hc = std::thread::hardware_concurrency();
    if (hc == 0) hc = 4;
    unsigned gpus = (unsigned)std::max<size_t>(1, n_devices_of_handle);
    if (const char *e = getenv("LOCAL_WORLD_SIZE")) gpus = std::max(gpus, (unsigned)std::max(1, atoi(e)));
    const double cores = std::max(1.0, std::min((double)hc / gpus, (double)host_threads())), r_host = 2.5 * cores, r_pcie = 24.0;
    host_share = std::min(0.9, r_host / (r_pcie + 0.73 * r_host));   // a host-packed base still sends 0.27 bytes
    const int set = g_pack_mode.load();
    const int forced = set > 0 ? set : (set < 0 ? env : 0);
    if (forced == kPackOnHost || forced == kPackOnDevice) return (PackMode)forced;
    if (forced == kPackMixed) return fast_plan ? kPackMixed : kPackOnDevice;
    return hc / gpus >= 16 ? kPackOnHost : kPackOnDevice;
}

static bool is_pinned_host(const void *p) {
    cudaPointerAttributes a{};
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { (void)cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost;
}

// Reads of a batch planned just in time (place_batch_impl, `fast`): the optimistic plan of a batch of short reads - every
// read has k .. 162 bases (one geometry of the scan kernel), so the device order is the input order, nothing is decided
// on the host, and the layout of a chunk (word offsets, lengths) is written right before the chunk is enqueued instead of
// in a pass over the whole batch before the first copy starts (0.7 ms per million reads on sixteen threads, 2.7 ms on
// four: SCALE_r01's end-to-end curve).  Returns false - nothing written beyond `end` - when a read does not qualify;
// the caller then starts over with the general plan (plan_batch).
constexpr uint32_t kFastMaxLen = 162;
static bool plan_reads_fast(const cls_batch *batch, uint32_t k, PackedLayout &lay, std::vector<uint32_t> &word_off, uint64_t first,
                            uint64_t end, uint64_t &words_so_far, uint32_t &max_len, ReadDesc *descs, uint64_t *src, uint64_t base0) {
    constexpr uint64_t kBlk = 8192;
    const uint64_t n = end - first, nblk = (n + kBlk - 1) / kBlk;
    std::vector<uint64_t> bw(nblk + 1, 0);
    std::vector<uint32_t> bmx(nblk, 0);
    std::atomic<bool> ok{true};
    parallel_for(nblk, 4, [&](uint64_t b0, uint64_t b1) {
        for (uint64_t blk = b0; blk < b1; ++blk) {
            uint64_t wsum = 0;
            uint32_t mx = 0;
            bool good = true;
            const uint64_t hi = std::min(end, first + (blk + 1) * kBlk);
            for (uint64_t i = first + blk * kBlk; i < hi; ++i) {
                const uint64_t o0 = batch->offsets[i], o1 = batch->offsets[i + 1];
                const uint64_t len = o1 - o0;
                good &= (o1 >= o0) & (len >= k) & (len <= kFastMaxLen);
                lay.lens[i] = (uint32_t)len;
                wsum += (len + 15u) / 16u;
                mx = std::max(mx, (uint32_t)std::min<uint64_t>(len, 0xFFFFFFFFu));
            }
            if (!good) ok = false;
            bw[blk + 1] = wsum;
            bmx[blk] = mx;
        }
    });
    if (!ok) return false;
    bw[0] = words_so_far;
    for (uint64_t b = 0; b < nblk; ++b) { bw[b + 1] += bw[b]; max_len = std::max(max_len, bmx[b]); }
    if (bw[nblk] >= 0xFFFFFFFFull) return false;   // the general plan reports it
    parallel_for(nblk, 4, [&](uint64_t b0, uint64_t b1) {
        for (uint64_t blk = b0; blk < b1; ++blk) {
            uint64_t wo = bw[blk];
            const uint64_t hi = std::min(end, first + (blk + 1) * kBlk);
            for (uint64_t i = first + blk * kBlk; i < hi; ++i) {
                lay.perm[i] = (uint32_t)i;
                lay.pre_status[i] = 0xFF;
                word_off[i] = (uint32_t)wo;
                descs[i] = ReadDesc{(uint32_t)wo, lay.lens[i]};
                if (src) src[i] = batch->offsets[i] - base0;   // device packing: where the read's bases start
                wo += (lay.lens[i] + 15u) / 16u;
            }
        }
    });
    words_so_far = bw[nblk];
    word_off[end] = (uint32_t)words_so_far;
    return true;
}

static int place_batch_impl(cls_index *ix, const cls_batch *batch, const cls_params *params, cls_result *result,
                            size_t n_devices_of_handle, bool fast, bool *fell_back) {
    const double t0 = now_ms();
    CU_TRY(cudaSetDevice(ix->device));
    Workspace *w = acquire_ws(ix);
    if (!w) return fail(CLS_ERR_CUDA, "could not create a stream/workspace");
    WsGuard guard{ix, w};
    PackedLayout &lay = w->lay;
    std::vector<uint32_t> &word_off = lay.word_off;
    int rc = CLS_OK;
    const uint64_t nq = batch->n_queries;
    uint64_t fast_words = 0;       // fast plan: packed words of the reads planned so far
    uint64_t fast_planned = 0;     //            ... and how many reads that is
    if (fast) {
        const uint64_t tb = batch->offsets[nq] - batch->offsets[0];
        lay.classes.clear();
        lay.n_queries = nq; lay.n_device = (uint32_t)nq;
        lay.n_words = (tb + 15 * nq) / 16 + 1;   // an upper bound, for the buffers
        lay.pre_status.resize(nq); lay.lens.resize(nq); lay.perm.resize(nq); word_off.resize((size_t)nq + 1);
        lay.classes.push_back(LengthClass{0, (uint32_t)nq, (uint32_t)std::min<uint64_t>(kFastMaxLen, std::max<uint64_t>(tb / nq, ix->dix.k_size))});
    } else {
        rc = plan_batch(batch, ix->dix.k_size, ix->dix.max_fanout, lay, word_off);
        if (rc != CLS_OK) return rc;
    }
    cls_timing tm{};
    tm.pack_ms = now_ms() - t0;  // planning counts as packing
    static const bool dbg = getenv("CLS_DEBUG_TIMING") != nullptr;
    if (dbg) fprintf(stderr, "[place_batch] plan %.2f ms\n", tm.pack_ms);
    const size_t words_b = (size_t)lay.n_words * 4, descs_b = (size_t)lay.n_device * sizeof(ReadDesc),
                 res_b = (size_t)lay.n_device * sizeof(ResultRec);
    PlaceParams pp = make_place_params(params);
    const uint64_t base0 = batch->n_queries ? batch->offsets[0] : 0;
    const uint64_t ascii_b = batch->n_queries ? batch->offsets[batch->n_queries] - base0 : 0;
    double host_share = 0.0;
    const PackMode pack_mode = lay.n_device && ascii_b ? resolve_pack_mode(n_devices_of_handle, fast, host_share) : kPackOnHost;
    const bool dev_pack = pack_mode != kPackOnHost, mix = pack_mode == kPackMixed;
    // the whole range must be pinned for a direct copy (first and last byte looked at; a registration covers a range)
    const bool src_pinned = dev_pack && is_pinned_host(batch->bases + base0) && is_pinned_host(batch->bases + base0 + ascii_b - 1);
    constexpr uint64_t kPiece = (uint64_t)32 << 20;   // bases per copy
    if (lay.n_device) {
        if (!dev_pack || mix) CU_TRY(w->h_words.reserve(words_b + 16));
        CU_TRY(w->h_descs.reserve(descs_b)); CU_TRY(w->h_results.reserve(res_b));
        CU_TRY(w->d_words.reserve(words_b + 16)); CU_TRY(w->d_descs.reserve(descs_b)); CU_TRY(w->d_results.reserve(res_b));
        if (dev_pack) {
            CU_TRY(w->d_ascii.reserve(ascii_b + 16)); CU_TRY(w->d_src.reserve((size_t)lay.n_device * 8)); CU_TRY(w->d_bad.reserve(lay.n_device));
            CU_TRY(w->h_src.reserve((size_t)lay.n_device * 8)); CU_TRY(w->h_bad.reserve(lay.n_device));
            if (!src_pinned)
                for (int q = 0; q < 2; ++q) {
                    CU_TRY(w->h_stage[q].reserve(std::min(kPiece, ascii_b)));
                    if (!w->stage_ev[q]) CU_TRY(cudaEventCreateWithFlags(&w->stage_ev[q], cudaEventDisableTiming));
                }
        }
    }
    // Chunks of every length class go through pack (host threads) -> H2D -> kernel -> D2H on three
    // streams: chunk c+1 is packed and copied while chunk c is on the SMs, and the
    // results of finished chunks are scattered to the caller's arrays while later chunks run.
    struct Chunk { uint32_t first, count, max_len; };
    std::vector<Chunk> chunks;
    // bases per chunk: 24 M (160 k reads of 150 bases), more for big batches - at least a twelfth of the batch, so that
    // the per-launch tails of the persistent kernels stay a small share of a chunk (CLS_CHUNK_MBASES fixes the size)
    static const uint64_t kChunkEnv = [] { const char *e = getenv("CLS_CHUNK_MBASES"); return (uint64_t)(e ? atoi(e) : 0) << 20; }();
    const uint64_t total_bases = batch->n_queries ? batch->offsets[batch->n_queries] - batch->offsets[0] : 0;
    const uint64_t kChunkBases = kChunkEnv ? kChunkEnv : std::max<uint64_t>((uint64_t)24 << 20, total_bases / 12);
    // the very first chunk holds a quarter of `per` reads so that the GPU starts early; later ones grow up to twice `per`
    // (fewer launch tails).  (x 1.5 per chunk: the host packs chunk c + 1 while the GPU places chunk c, at about half the
    // GPU's time per read - doubling the chunks left the GPU waiting at every step of the ramp: 54.8 against 52.2 ms per
    // 10 M reads, profiles/r2b)
    constexpr uint64_t kFirstChunkDiv = 4, kChunkGrowthPct = 150, kChunkRampMax = 2;
    for (const LengthClass &c : lay.classes) {
        const uint64_t per = std::max<uint64_t>(4096, kChunkBases / std::max<uint32_t>(c.max_len, 1));
        uint64_t a = 0, step = chunks.empty() ? std::max<uint64_t>(4096, per / kFirstChunkDiv) : per;
        while (a < c.count) {
            const uint64_t n = std::min<uint64_t>(step, c.count - a);
            chunks.push_back(Chunk{(uint32_t)(c.first + a), (uint32_t)n, c.max_len});
            a += n;
            step = std::min<uint64_t>(step * kChunkGrowthPct / 100, per * kChunkRampMax);
        }
        // ... and the very last ones shrink again: what follows the last kernel (its results' way back, their scatter) is
        // exposed, and is as long as the last chunk
        if (&c == &lay.classes.back())
            for (int r = 0; r < 3 && chunks.back().count > std::max<uint64_t>(8192, per / 4); ++r) {
                Chunk last = chunks.back();
                const uint32_t half = last.count / 2;
                chunks.back().count = last.count - half;
                chunks.push_back(Chunk{last.first + (last.count - half), half, last.max_len});
            }
    }
    while (w->chunk_ev.size() < 4 * chunks.size()) {
        cudaEvent_t e = nullptr;
        CU_TRY(cudaEventCreate(&e));
        w->chunk_ev.push_back(e);
    }
    uint32_t *h_words = (uint32_t *)w->h_words.p, *d_words = (uint32_t *)w->d_words.p;
    ReadDesc *h_descs = (ReadDesc *)w->h_descs.p, *d_descs = (ReadDesc *)w->d_descs.p;
    ResultRec *h_res = (ResultRec *)w->h_results.p, *d_res = (ResultRec *)w->d_results.p;
    uint64_t *h_src = (uint64_t *)w->h_src.p, *d_src = (uint64_t *)w->d_src.p;
    uint8_t *h_bad = (uint8_t *)w->h_bad.p, *d_bad = (uint8_t *)w->d_bad.p, *d_ascii = (uint8_t *)w->d_ascii.p;
    size_t scattered = 0;
    uint64_t host_done = 0;                              // queries (caller order) whose host-decided fields are written
    std::vector<uint8_t> chunk_dev(chunks.size(), 0);   // chunk packed on the device (its invalid-base flags come back with the results)
    double host_acc = 0.5;                               // mixed: error diffusion of the host's share over the chunks
    auto drain = [&](size_t upto) -> int {  // scatter the chunks whose D2H has completed (blocking up to `upto`)
        for (; scattered < upto; ++scattered) {
            CU_TRY(cudaEventSynchronize(w->chunk_ev[4 * scattered + 3]));
            scatter_device_range(lay, h_res, result, chunks[scattered].first, chunks[scattered].count, chunk_dev[scattered] ? h_bad : nullptr);
        }
        return CLS_OK;
    };
    // Copies in, kernels and copies out run on THREE streams chained by events, so that the kernels of consecutive
    // chunks never share the SMs (with everything of a chunk on one of two alternating streams the scan kernel of chunk
    // c + 1 starts while the descent kernel of chunk c still holds warp slots: 8.13 against 7.70 ms per 1 M reads end to
    // end, profiles/r2a).
    // With device packing the bases go up in pieces that do not end where the chunks end: a piece copied for chunk c holds
    // the first bases of chunk c + 1, so all copies in have to share ONE stream for a chunk's pack kernel to wait for them.
    cudaStream_t st_in = w->stream2, st_k = w->stream, st_out = w->stream3;
    // device packing: the caller's bases go up in input order, piece by piece, on the copy stream; a chunk's pack kernel
    // runs once everything up to the last base of its reads is there (one length class: chunk c needs just its own range)
    uint64_t uploaded = 0, piece_no = 0;
    auto upload_to = [&](uint64_t end) -> int {
        while (uploaded < end) {
            const uint64_t n = std::min(kPiece, end - uploaded);
            const uint8_t *src = batch->bases + base0 + uploaded;
            if (!src_pinned) {
                const int q = (int)(piece_no & 1);
                if (piece_no >= 2) CU_TRY(cudaEventSynchronize(w->stage_ev[q]));   // the copy that last read this slot
                uint8_t *dst = (uint8_t *)w->h_stage[q].p;
                parallel_for(n, (uint64_t)1 << 20, [&](uint64_t a, uint64_t b) { memcpy(dst + a, src + a, b - a); });
                src = dst;
                CU_TRY(cudaMemcpyAsync(d_ascii + uploaded, src, n, cudaMemcpyHostToDevice, st_in));
                CU_TRY(cudaEventRecord(w->stage_ev[q], st_in));
            } else {
                CU_TRY(cudaMemcpyAsync(d_ascii + uploaded, src, n, cudaMemcpyHostToDevice, st_in));
            }
            tm.h2d_bytes += n;
            uploaded += n; ++piece_no;
        }
        return CLS_OK;
    };
    for (size_t ci = 0; ci < chunks.size(); ++ci) {
        if (fast) {   // the layout of this chunk's reads, just in time
            const double tq = now_ms();
            uint32_t mx = 0;
            const uint64_t end = (uint64_t)chunks[ci].first + chunks[ci].count;
            if (!plan_reads_fast(batch, ix->dix.k_size, lay, word_off, fast_planned, end, fast_words, mx, h_descs, dev_pack ? h_src : nullptr, base0)) {
                // a read that is too short, too long or has bad offsets: everything in flight is waited for (the guard),
                // and the caller starts over with the general plan
                *fell_back = true;
                return CLS_OK;
            }
            fast_planned = end;
            chunks[ci].max_len = mx;
            tm.pack_ms += now_ms() - tq;
        }
        const Chunk &c = chunks[ci];
        cudaEvent_t *ev = &w->chunk_ev[4 * ci];
        const double tp = now_ms();
        const size_t w0 = word_off[c.first], w1 = word_off[c.first + c.count];
        bool dev_c = dev_pack;
        if (mix) {
            host_acc += host_share;
            if (host_acc >= 1.0) { host_acc -= 1.0; dev_c = false; }
        }
        chunk_dev[ci] = dev_c ? 1 : 0;
        if (dev_c) {
            // descriptors and source offsets of the chunk's reads; how far into the bases the chunk reaches
            // (the just-in-time plan has written them already, and the chunk's bases are one range)
            std::atomic<uint64_t> need{fast ? batch->offsets[(uint64_t)c.first + c.count] - base0 : 0};
            if (!fast) parallel_for(c.count, 16384, [&](uint64_t a0, uint64_t b0) {
                uint64_t mx = 0;
                for (uint64_t j = c.first + a0; j < c.first + b0; ++j) {
                    const uint64_t i = lay.perm[j];
                    h_descs[j] = ReadDesc{word_off[j], lay.lens[i]};
                    h_src[j] = batch->offsets[i] - base0;
                    mx = std::max(mx, batch->offsets[i + 1] - base0);
                }
                uint64_t cur = need.load();
                while (cur < mx && !need.compare_exchange_weak(cur, mx)) {}
            });
            CU_TRY(cudaEventRecord(ev[0], st_in));
            CU_TRY(cudaMemsetAsync(d_bad + c.first, 0, c.count, st_in));
            // (just-in-time plan: the device order is the input order, a chunk's bases are one range - the ranges of
            // host-packed chunks are never sent)
            if (fast && uploaded < h_src[c.first]) uploaded = h_src[c.first];
            rc = upload_to(need.load());
            if (rc != CLS_OK) return rc;
            tm.pack_ms += now_ms() - tp;
            CU_TRY(cudaMemcpyAsync(d_src + c.first, h_src + c.first, (size_t)c.count * 8, cudaMemcpyHostToDevice, st_in));
            tm.h2d_bytes += (uint64_t)c.count * 8;
        } else {
            pack_batch(batch, lay, word_off, h_words, h_descs, c.first, c.count);
            tm.pack_ms += now_ms() - tp;
            CU_TRY(cudaEventRecord(ev[0], st_in));
            CU_TRY(cudaMemcpyAsync(d_words + w0, h_words + w0, (w1 - w0) * 4, cudaMemcpyHostToDevice, st_in));
            tm.h2d_bytes += (w1 - w0) * 4;
        }
        CU_TRY(cudaMemcpyAsync(d_descs + c.first, h_descs + c.first, (size_t)c.count * sizeof(ReadDesc), cudaMemcpyHostToDevice, st_in));
        tm.h2d_bytes += (uint64_t)c.count * sizeof(ReadDesc);
        CU_TRY(cudaEventRecord(ev[1], st_in));
        CU_TRY(cudaStreamWaitEvent(st_k, ev[1], 0));
        if (dev_c) {
            cudaError_t pe = launch_ascii_pack(d_ascii, d_src, d_descs, c.first, c.count, c.max_len, d_words, d_bad, st_k);
            if (pe != cudaSuccess) return fail(CLS_ERR_CUDA, std::string("pack kernel launch: ") + cudaGetErrorString(pe));
            tm.kernel_launches += 1;
        }
        PlaceGeom g = make_place_geom(c.max_len, ix->dix.k_size, ix->dix.max_fanout);
        DevBuf &scratch = w->d_scratch;
        const size_t scratch_b = place_scratch_bytes(c.count, c.max_len, ix->dix.k_size, ix->dix.max_fanout);
        if (scratch_b > scratch.cap && scratch.p)
            CU_TRY(cudaStreamSynchronize(st_k));   // growing the scratch buffer frees it: nothing on the kernel stream may still use it
        CU_TRY(scratch.reserve(scratch_b));
        uint32_t nl = 0;
        cudaError_t e = launch_place(ix->dix, pp, d_words, d_descs, c.first, c.count, d_res, g, ix->sm_count, st_k,
                                     scratch.p, scratch.cap, &nl);
        if (e != cudaSuccess) {
            for (cudaStream_t s : {st_in, st_k, st_out}) cudaStreamSynchronize(s);
            if (e == cudaErrorInvalidConfiguration)
                return fail(CLS_ERR_UNSUPPORTED, "query too long (or tree fan-out too large) for the per-read shared-memory tables");
            return fail(CLS_ERR_CUDA, std::string("place kernel launch: ") + cudaGetErrorString(e));
        }
        tm.kernel_launches += nl;
        CU_TRY(cudaEventRecord(ev[2], st_k));
        CU_TRY(cudaStreamWaitEvent(st_out, ev[2], 0));
        CU_TRY(cudaMemcpyAsync(h_res + c.first, d_res + c.first, (size_t)c.count * sizeof(ResultRec), cudaMemcpyDeviceToHost, st_out));
        tm.d2h_bytes += (uint64_t)c.count * sizeof(ResultRec);
        if (dev_c) {
            CU_TRY(cudaMemcpyAsync(h_bad + c.first, d_bad + c.first, c.count, cudaMemcpyDeviceToHost, st_out));
            tm.d2h_bytes += c.count;
        }
        CU_TRY(cudaEventRecord(ev[3], st_out));
        if (ci >= 2) { rc = drain(ci - 1); if (rc != CLS_OK) return rc; }  // chunks older than the two in flight
        // fields decided on the host (n_query_kmers of every query; queries that never reach the device), a piece of the
        // caller's arrays per chunk - while the GPU has work, not in one pass after the last enqueue, where the last,
        // small chunks leave the GPU before a pass over ten million queries ends.  Just-in-time plan: the reads planned so
        // far (their lengths are known); general plan: an equal share per chunk.  A query demoted by a packer later on
        // (invalid base) is written again by the scatter of its chunk.
        const uint64_t upto = fast ? fast_planned : (uint64_t)((long double)nq * (ci + 1) / chunks.size());
        scatter_host_decided(lay, ix->dix.k_size, result, host_done, upto);
        host_done = std::max(host_done, std::min(upto, nq));
    }
    const double th = now_ms();
    scatter_host_decided(lay, ix->dix.k_size, result, host_done, nq);   // what is left (all of it when nothing reaches the device)
    if (dbg) fprintf(stderr, "[place_batch] enqueue done at %.2f ms, host-decided fields %.2f ms\n", th - t0, now_ms() - th);
    rc = drain(chunks.size());
    if (rc != CLS_OK) return rc;
    if (dbg) fprintf(stderr, "[place_batch] drained at %.2f ms\n", now_ms() - t0);
    for (size_t ci = 0; ci < chunks.size(); ++ci) {
        float ms = 0;
        cudaEvent_t *ev = &w->chunk_ev[4 * ci];
        cudaEventElapsedTime(&ms, ev[0], ev[1]); tm.h2d_ms += ms;
        cudaEventElapsedTime(&ms, ev[1], ev[2]); tm.kernel_ms += ms;
        cudaEventElapsedTime(&ms, ev[2], ev[3]); tm.d2h_ms += ms;
    }
    tm.total_ms = now_ms() - t0;
    tm.pack_on_device = mix ? 3u : dev_pack ? (src_pinned ? 2u : 1u) : 0u;
    { std::lock_guard<std::mutex> lk(ix->mu); ix->timing = tm; }
    guard.clean = true;   // every chunk has been drained: nothing of this call is in flight
    return CLS_OK;
}

static int place_batch_one(cls_index *ix, const cls_batch *batch, const cls_params *params, cls_result *result,
                           size_t n_devices_of_handle = 1) {
    if (ix->n_shards > 1) return fail(CLS_ERR_INVALID_ARGUMENT, "this handle holds one shard of the index: use the routed calls");
    // batches that look like short reads (k = 35, mean length within the one-warp geometry) try the just-in-time plan
    const uint64_t n = batch->n_queries;
    bool fast = ix->dix.k_size == 35 && n >= 1 && n < 0xFFFFFFFFull && batch->offsets && batch->bases;
    if (fast) {
        const uint64_t o0 = batch->offsets[0], o1 = batch->offsets[n];
        fast = o1 >= o0 && (o1 - o0) >= n * 35 && (o1 - o0) <= n * (uint64_t)kFastMaxLen;
    }
    if (fast) {
        bool fell_back = false;
        const int rc = place_batch_impl(ix, batch, params, result, n_devices_of_handle, true, &fell_back);
        if (!fell_back) return rc;
    }
    bool unused = false;
    return place_batch_impl(ix, batch, params, result, n_devices_of_handle, false, &unused);
}

// Cut points of a batch into `nd` contiguous parts of equal shares of the bases (cut[0] = 0, cut[nd] = n).
static std::vector<uint64_t> cut_by_bases(const cls_batch *batch, size_t nd) {
    const uint64_t n = batch->n_queries;
    std::vector<uint64_t> cut(nd + 1, n);
    cut[0] = 0;
    if (n) {
        const uint64_t b0 = batch->offsets[0], total = batch->offsets[n] >= b0 ? batch->offsets[n] - b0 : 0;
        for (size_t d = 1; d < nd; ++d) {
            const uint64_t want = b0 + (uint64_t)((long double)total * d / nd);
            uint64_t lo = cut[d - 1], hi = n;      // first query starting at or after `want` (offsets are checked per part)
            while (lo < hi) { const uint64_t mid = (lo + hi) / 2; if (batch->offsets[mid] < want) lo = mid + 1; else hi = mid; }
            cut[d] = lo;
        }
    }
    return cut;
}

// The caller's result arrays from query `a` on.
static cls_result result_from(const cls_result *result, uint64_t a) {
    cls_result r{};
    r.status = result->status ? result->status + a : nullptr;
    r.node_id = result->node_id ? result->node_id + a : nullptr;
    r.one = result->one ? result->one + a : nullptr;
    r.rest = result->rest ? result->rest + a : nullptr;
    r.n_query_kmers = result->n_query_kmers ? result->n_query_kmers + a : nullptr;
    r.n_matched = result->n_matched ? result->n_matched + a : nullptr;
    r.n_root_matched = result->n_root_matched ? result->n_root_matched + a : nullptr;
    r.iterations = result->iterations ? result->iterations + a : nullptr;
    return r;
}

// Multi-device handle: the batch is cut into one contiguous part per replica (equal shares of the bases), every part
// goes through the single-device pipeline on its own host thread (the packing loops of all parts share the one host
// pool), and the result arrays are written in place - the reference's single process fanning out over its workers
// (ports/cli/src/cmds/place_sequences.rs:125-156, place_sequences/mod.rs:123-126).
static int place_batch_multi(cls_index *front, const cls_batch *batch, const cls_params *params, cls_result *result) {
    const size_t nd = front->replicas.size();
    const uint64_t n = batch->n_queries;
    if (n && !batch->offsets) return fail(CLS_ERR_INVALID_ARGUMENT, "batch arrays are NULL");
    const std::vector<uint64_t> cut = cut_by_bases(batch, nd);
    std::vector<int> rcs(nd, CLS_OK);
    std::vector<std::string> errs(nd);
    auto run = [&](size_t d) {
        const uint64_t a = cut[d], cnt = cut[d + 1] - a;
        if (cnt == 0) return;
        const cls_batch part{cnt, batch->bases, batch->offsets + a};   // offsets are absolute into `bases`
        cls_result r = result_from(result, a);
        try {
            rcs[d] = place_batch_one(front->replicas[d].get(), &part, params, &r, nd);
        } catch (const std::bad_alloc &) {
            rcs[d] = fail(CLS_ERR_OUT_OF_MEMORY, "host allocation failed");
        } catch (const std::exception &e) {
            rcs[d] = fail(CLS_ERR_INVALID_ARGUMENT, e.what());
        }
        if (rcs[d] != CLS_OK) errs[d] = g_last_error;   // thread-local: carry it to the caller's thread
    };
    std::vector<std::thread> th;
    for (size_t d = 1; d < nd; ++d) th.emplace_back(run, d);
    run(0);
    for (auto &t : th) t.join();
    cls_timing tm{};
    for (size_t d = 0; d < nd; ++d) {
        std::lock_guard<std::mutex> lk(front->replicas[d]->mu);
        const cls_timing &t = front->replicas[d]->timing;
        tm.pack_ms = std::max(tm.pack_ms, t.pack_ms); tm.h2d_ms = std::max(tm.h2d_ms, t.h2d_ms);
        tm.kernel_ms = std::max(tm.kernel_ms, t.kernel_ms); tm.d2h_ms = std::max(tm.d2h_ms, t.d2h_ms);
        tm.total_ms = std::max(tm.total_ms, t.total_ms); tm.kernel_launches += t.kernel_launches;
        tm.h2d_bytes += t.h2d_bytes; tm.d2h_bytes += t.d2h_bytes; tm.pack_on_device = std::max(tm.pack_on_device, t.pack_on_device);
    }
    { std::lock_guard<std::mutex> lk(front->mu); front->timing = tm; }
    for (size_t d = 0; d < nd; ++d)
        if (rcs[d] != CLS_OK) return fail(rcs[d], errs[d]);
    return CLS_OK;
}

int cls_set_pack_mode(int mode) {
    if (mode < 0 || mode > 3) return fail(CLS_ERR_INVALID_ARGUMENT, "pack mode must be 0 (automatic), 1 (host), 2 (device) or 3 (mixed)");
    const int prev = g_pack_mode.exchange(mode);
    return prev < 0 ? 0 : prev;
}

int cls_place_batch(cls_index *ix, const cls_batch *batch, const cls_params *params, cls_result *result) try {
    if (!ix || !batch || !params || !result) return fail(CLS_ERR_INVALID_ARGUMENT, "NULL argument");
    if (ix->sharded) return ix->sharded->place_batch(ix, batch, params, result);
    if (!ix->replicas.empty()) return place_batch_multi(ix, batch, params, result);
    return place_batch_one(ix, batch, params, result);
} CLS_ABI_CATCH

int cls_batch_upload(cls_index *ix, const cls_batch *batch, cls_resident_batch **out) try {
    if (!ix || !batch || !out) return fail(CLS_ERR_INVALID_ARGUMENT, "NULL argument");
    if (!ix->shards.empty()) ix = ix->shards[0].get();       // a sharded handle: resident batches live on its first shard's device
    if (!ix->replicas.empty()) ix = ix->replicas[0].get();   // a multi-device handle: resident batches live on its first device
    *out = nullptr;
    CU_TRY(cudaSetDevice(ix->device));
    auto rb = std::make_unique<cls_resident_batch>();
    rb->device = ix->device;
    std::vector<uint32_t> word_off;
    int rc = plan_batch(batch, ix->dix.k_size, ix->dix.max_fanout, rb->lay, word_off);
    if (rc != CLS_OK) return rc;
    const PackedLayout &lay = rb->lay;
    const size_t words_b = (size_t)lay.n_words * 4, descs_b = (size_t)lay.n_device * sizeof(ReadDesc),
                 res_b = (size_t)lay.n_device * sizeof(ResultRec);
    std::vector<uint32_t> words(lay.n_words + 4);
    std::vector<ReadDesc> descs(lay.n_device);
    pack_batch(batch, rb->lay, word_off, words.data(), descs.data());
    CU_TRY(rb->d_words.reserve(words_b + 16)); CU_TRY(rb->d_descs.reserve(descs_b + 16)); CU_TRY(rb->d_results.reserve(res_b + 32));
    CU_TRY(rb->h_results.reserve(res_b + 32));
    CU_TRY(cudaMemcpy(rb->d_words.p, words.data(), words_b, cudaMemcpyHostToDevice));
    CU_TRY(cudaMemcpy(rb->d_descs.p, descs.data(), descs_b, cudaMemcpyHostToDevice));
    CU_TRY(cudaMemset(rb->d_results.p, 0xFF, res_b));
    *out = rb.release();
    return CLS_OK;
} CLS_ABI_CATCH

// The tail of both text ingests: the records' lengths are in rb->fa_length and their first kept base in `src`; plan them
// with the planner of cls_batch_upload and pack them from the compacted codes on the device.
static int pack_ingested(cls_index *ix, cls_resident_batch *rb, const uint8_t *d_codes, const std::vector<uint64_t> &src, cudaStream_t st) {
    const auto &ln = rb->fa_length;
    const uint64_t n = ln.size();
    std::vector<uint64_t> offsets(n + 1, 0);
    for (uint64_t i = 0; i < n; ++i) offsets[i + 1] = offsets[i] + ln[i];
    cls_batch fake{n, reinterpret_cast<const uint8_t *>(offsets.data()), offsets.data()};   // plan_batch never reads the bases
    std::vector<uint32_t> word_off;
    int rc = plan_batch(&fake, ix->dix.k_size, ix->dix.max_fanout, rb->lay, word_off);
    if (rc != CLS_OK) return rc;
    const PackedLayout &lay = rb->lay;
    const size_t words_b = (size_t)lay.n_words * 4, descs_b = (size_t)lay.n_device * sizeof(ReadDesc), res_b = (size_t)lay.n_device * sizeof(ResultRec);
    CU_TRY(rb->d_words.reserve(words_b + 16)); CU_TRY(rb->d_descs.reserve(descs_b + 16)); CU_TRY(rb->d_results.reserve(res_b + 32));
    if (lay.n_device) {   // the pinned result buffer is allocated by the first cls_resident_fetch
        DevBuf d_src, d_woff, d_len;
        struct Free { std::vector<DevBuf *> b; ~Free() { for (auto *x : b) x->release(); } } guard{{&d_src, &d_woff, &d_len}};
        std::vector<ReadDesc> descs(lay.n_device);
        std::vector<uint64_t> src_dev(lay.n_device);
        std::vector<uint32_t> len_dev(lay.n_device);
        parallel_for(lay.n_device, 1 << 15, [&](uint64_t j0, uint64_t j1) {
            for (uint64_t j = j0; j < j1; ++j) {
                const uint32_t i = lay.perm[j];
                descs[j] = ReadDesc{word_off[j], ln[i]};
                src_dev[j] = src[i];
                len_dev[j] = ln[i];
            }
        });
        CU_TRY(d_src.reserve(src_dev.size() * 8)); CU_TRY(d_woff.reserve(word_off.size() * 4)); CU_TRY(d_len.reserve(len_dev.size() * 4));
        CU_TRY(cudaMemcpyAsync(d_src.p, src_dev.data(), src_dev.size() * 8, cudaMemcpyHostToDevice, st));
        CU_TRY(cudaMemcpyAsync(d_woff.p, word_off.data(), (size_t)lay.n_device * 4, cudaMemcpyHostToDevice, st));
        CU_TRY(cudaMemcpyAsync(d_len.p, len_dev.data(), len_dev.size() * 4, cudaMemcpyHostToDevice, st));
        CU_TRY(cudaMemcpyAsync(rb->d_descs.p, descs.data(), descs_b, cudaMemcpyHostToDevice, st));
        CU_TRY(launch_fasta_pack(d_codes, (const uint64_t *)d_src.p, (const uint32_t *)d_woff.p, (const uint32_t *)d_len.p,
                                 lay.n_device, (uint32_t *)rb->d_words.p, ix->sm_count, st));
        CU_TRY(cudaMemsetAsync(rb->d_results.p, 0xFF, res_b, st));
        CU_TRY(cudaStreamSynchronize(st));
    }
    return CLS_OK;
}

// ---- FASTA ingest on the device (SURVEY.md section 8f row 3; file_or_stdin.rs:76-116, sequence.rs:47-56) -----------
int cls_fasta_upload(cls_index *ix, const uint8_t *text, uint64_t n_bytes, cls_resident_batch **out, cls_fasta_records *records) try {
    if (!ix || !out || !records || (n_bytes && !text)) return fail(CLS_ERR_INVALID_ARGUMENT, "NULL argument");
    if (!ix->shards.empty()) ix = ix->shards[0].get();       // a sharded handle: resident batches live on its first shard's device
    if (!ix->replicas.empty()) ix = ix->replicas[0].get();   // a multi-device handle: resident batches live on its first device
    *out = nullptr;
    std::memset(records, 0, sizeof *records);
    if (n_bytes >= (1ull << 32)) return fail(CLS_ERR_UNSUPPORTED, "FASTA text of 4 GiB or more: split it (the tile summaries count in 32 bits)");
    CU_TRY(cudaSetDevice(ix->device));
    static const bool dbg = getenv("CLS_DEBUG_TIMING") != nullptr;
    double tlast = now_ms();
    auto lap = [&](const char *what) { if (dbg) { const double t = now_ms(); fprintf(stderr, "[fasta] %-22s %8.2f ms\n", what, t - tlast); tlast = t; } };
    auto rb = std::make_unique<cls_resident_batch>();
    rb->device = ix->device;
    cudaStream_t st = nullptr;
    DevBuf d_text, d_tiles, d_bases, d_misc, d_codes, d_hpos, d_hkept, d_hflag;
    struct Free { std::vector<DevBuf *> b; ~Free() { for (auto *x : b) x->release(); } }
        guard{{&d_text, &d_tiles, &d_bases, &d_misc, &d_codes, &d_hpos, &d_hkept, &d_hflag}};
    const uint32_t nt = fasta_n_tiles(n_bytes);
    TileBase totals{0, 0, 0, 0};
    uint32_t non_ascii = 0;
    if (n_bytes) {
        CU_TRY(d_text.reserve(n_bytes + 16)); CU_TRY(d_tiles.reserve((size_t)nt * fasta_tile_bytes())); CU_TRY(d_bases.reserve((size_t)nt * sizeof(TileBase)));
        CU_TRY(d_misc.reserve(256));
        lap("alloc");
        CU_TRY(cudaMemcpyAsync(d_text.p, text, n_bytes, cudaMemcpyHostToDevice, st));
        CU_TRY(cudaMemsetAsync(d_misc.p, 0, 256, st));
        TileBase *d_totals = (TileBase *)d_misc.p;
        uint32_t *d_non_ascii = (uint32_t *)((char *)d_misc.p + 128);
        CU_TRY(launch_fasta_scan((const uint8_t *)d_text.p, n_bytes, d_tiles.p, (TileBase *)d_bases.p, d_totals, d_non_ascii, st));
        CU_TRY(cudaMemcpyAsync(&totals, d_totals, sizeof totals, cudaMemcpyDeviceToHost, st));
        CU_TRY(cudaMemcpyAsync(&non_ascii, d_non_ascii, 4, cudaMemcpyDeviceToHost, st));
        CU_TRY(cudaStreamSynchronize(st));
        lap("h2d + scan");
    }
    if (non_ascii)
        return fail(CLS_ERR_UNSUPPORTED, "non-ASCII byte in the FASTA text: Rust's to_uppercase() is Unicode-aware - use the host reader for this file");
    const uint64_t n_hdr = totals.hdrs, n_kept = totals.kept;
    if (n_hdr >= 0xFFFFFFFFull) return fail(CLS_ERR_UNSUPPORTED, "more than 2^32-1 header lines");
    std::vector<uint64_t> hpos(n_hdr), hkept(n_hdr);
    std::vector<uint32_t> hflag(n_hdr);
    if (n_hdr || n_kept) {
        CU_TRY(d_codes.reserve(n_kept + 16)); CU_TRY(d_hpos.reserve(n_hdr * 8 + 8)); CU_TRY(d_hkept.reserve(n_hdr * 8 + 8)); CU_TRY(d_hflag.reserve(n_hdr * 4 + 4));
        CU_TRY(cudaMemsetAsync(d_hflag.p, 0, n_hdr * 4 + 4, st));
        CU_TRY(launch_fasta_write((const uint8_t *)d_text.p, n_bytes, (const TileBase *)d_bases.p, (uint8_t *)d_codes.p, (uint64_t *)d_hpos.p,
                                  (uint64_t *)d_hkept.p, (uint32_t *)d_hflag.p, st));
        if (n_hdr) {
            CU_TRY(cudaMemcpyAsync(hpos.data(), d_hpos.p, n_hdr * 8, cudaMemcpyDeviceToHost, st));
            CU_TRY(cudaMemcpyAsync(hkept.data(), d_hkept.p, n_hdr * 8, cudaMemcpyDeviceToHost, st));
            CU_TRY(cudaMemcpyAsync(hflag.data(), d_hflag.p, n_hdr * 4, cudaMemcpyDeviceToHost, st));
        }
        CU_TRY(cudaStreamSynchronize(st));
        lap("write + d2h");
    }
    // ---- the record rules of the reader (file_or_stdin.rs:91-113) on the per-header-line facts -----------------
    std::vector<uint64_t> src;      // first kept base of every record that is sent
    auto &hb = rb->fa_header_begin;
    auto &he = rb->fa_header_end;
    auto &ln = rb->fa_length;
    hb.reserve(n_hdr); src.reserve(n_hdr); ln.reserve(n_hdr);
    const bool orphan_sequence = n_hdr && hkept[0] > 0;   // bases before the first header: the reader errors out at that header (:96-100)
    if (n_hdr && !orphan_sequence) {
        for (uint64_t j = 0; j < n_hdr; ++j) {
            const bool last = j + 1 == n_hdr;
            const uint64_t kept = (last ? n_kept : hkept[j + 1]) - hkept[j];
            if (kept >= (1ull << 31)) return fail(CLS_ERR_INVALID_ARGUMENT, "query longer than 2^31 bases");
            if (!hflag[j]) {                    // header text empty after removing '>': the reader holds no header
                if (kept && !last) break;       // ... and errors out at the next header line (:96-100)
                continue;
            }
            if (last && kept == 0) continue;    // trailing record without sequence is dropped (:111-113)
            hb.push_back(hpos[j]);
            src.push_back(hkept[j]);
            ln.push_back((uint32_t)kept);
        }
    }
    lap("record rules");
    const uint64_t n = hb.size();
    he.resize(n);
    parallel_for(n, 4096, [&](uint64_t a, uint64_t b) {   // end of the header line's content: "\n" or "\r\n" excluded
        for (uint64_t i = a; i < b; ++i) {
            const uint8_t *s = text + hb[i];
            const void *nl = std::memchr(s, '\n', n_bytes - hb[i]);
            uint64_t e = nl ? (uint64_t)((const uint8_t *)nl - text) : n_bytes;
            if (nl && e > hb[i] && text[e - 1] == '\r') --e;
            he[i] = e;
        }
    });
    lap("header ends");
    const int rc = pack_ingested(ix, rb.get(), (const uint8_t *)d_codes.p, src, st);
    if (rc != CLS_OK) return rc;
    lap("pack");
    records->n_records = n;
    records->header_begin = hb.data();
    records->header_end = he.data();
    records->length = ln.data();
    *out = rb.release();
    return CLS_OK;
} CLS_ABI_CATCH

// ---- for the FASTQ ingest (fastq_ingest.cpp): the handle a resident batch of `ix` lives on, and the batch built from the
//      records a text ingest found (their first kept base `src` in the compacted codes on that device) -----------------------
}  // extern "C"
namespace cls {
cls_index *ingest_home(cls_index *ix, int *device, int *sm_count) {
    if (!ix->shards.empty()) ix = ix->shards[0].get();       // a sharded handle: resident batches live on its first shard's device
    if (!ix->replicas.empty()) ix = ix->replicas[0].get();   // a multi-device handle: resident batches live on its first device
    *device = ix->device;
    *sm_count = ix->sm_count;
    return ix;
}

int ingest_finish(cls_index *home, const uint8_t *d_codes, std::vector<uint64_t> &hb, std::vector<uint64_t> &he, std::vector<uint32_t> &ln,
                  const std::vector<uint64_t> &src, cudaStream_t st, cls_resident_batch **out, cls_fasta_records *records) try {
    auto rb = std::make_unique<cls_resident_batch>();
    rb->device = home->device;
    rb->fa_header_begin.swap(hb);
    rb->fa_header_end.swap(he);
    rb->fa_length.swap(ln);
    const int rc = pack_ingested(home, rb.get(), d_codes, src, st);
    if (rc != CLS_OK) return rc;
    records->n_records = rb->fa_length.size();
    records->header_begin = rb->fa_header_begin.data();
    records->header_end = rb->fa_header_end.data();
    records->length = rb->fa_length.data();
    *out = rb.release();
    return CLS_OK;
} CLS_ABI_CATCH
}  // namespace cls
extern "C" {

int cls_place_resident(cls_index *ix, cls_resident_batch *rb, const cls_params *params, void *stream) try {
    if (!ix || !rb || !params) return fail(CLS_ERR_INVALID_ARGUMENT, "NULL argument");
    if (ix->sharded) return ix->sharded->place_resident(ix, rb, params, (cudaStream_t)stream);
    if (!ix->replicas.empty()) ix = ix->replicas[0].get();   // a multi-device handle: resident batches live on its first device
    if (rb->device != ix->device) return fail(CLS_ERR_INVALID_ARGUMENT, "resident batch lives on another device");
    if (ix->n_shards > 1) return fail(CLS_ERR_INVALID_ARGUMENT, "this handle holds one shard of the index: use the routed calls");
    CU_TRY(cudaSetDevice(ix->device));
    uint64_t launches = 0;
    int rc = launch_classes(ix, rb->lay, params, (const uint32_t *)rb->d_words.p, (const ReadDesc *)rb->d_descs.p,
                            (ResultRec *)rb->d_results.p, (cudaStream_t)stream, rb->d_scratch, &launches);
    if (rc == CLS_OK) { std::lock_guard<std::mutex> lk(ix->mu); ix->timing.kernel_launches = launches; }
    return rc;
} CLS_ABI_CATCH

int cls_resident_fetch(cls_index *ix, cls_resident_batch *rb, void *stream, cls_result *result) try {
    if (!ix || !rb || !result) return fail(CLS_ERR_INVALID_ARGUMENT, "NULL argument");
    if (!ix->shards.empty()) ix = ix->shards[0].get();       // a sharded handle: resident batches live on its first shard's device
    if (!ix->replicas.empty()) ix = ix->replicas[0].get();   // a multi-device handle: resident batches live on its first device
    CU_TRY(cudaSetDevice(ix->device));
    const size_t res_b = (size_t)rb->lay.n_device * sizeof(ResultRec);
    if (res_b) {
        CU_TRY(rb->h_results.reserve(res_b + 32));
        CU_TRY(cudaMemcpyAsync(rb->h_results.p, rb->d_results.p, res_b, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    }
    CU_TRY(cudaStreamSynchronize((cudaStream_t)stream));
    scatter_results(rb->lay, ix->dix.k_size, (const ResultRec *)rb->h_results.p, result);
    return CLS_OK;
} CLS_ABI_CATCH

void cls_resident_destroy(cls_resident_batch *rb) { delete rb; }

uint64_t cls_resident_bytes(const cls_resident_batch *rb) {
    if (!rb) return 0;
    return (uint64_t)rb->lay.n_words * 4 + (uint64_t)rb->lay.n_device * (sizeof(ReadDesc) + sizeof(ResultRec));
}

// ---- hash-sharded index: route -> (all-to-all) -> probe -> (all-to-all) -> place --------------------
int cls_routed_windows(cls_index *ix, cls_resident_batch *rb, uint64_t *n_windows) try {
    if (!ix || !rb || !n_windows) return fail(CLS_ERR_INVALID_ARGUMENT, "NULL argument");
    if (!ix->shards.empty()) return fail(CLS_ERR_INVALID_ARGUMENT, "a sharded handle routes internally: the routed calls take the handle of one shard");
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
    if (!ix->shards.empty()) return fail(CLS_ERR_INVALID_ARGUMENT, "a sharded handle routes internally: the routed calls take the handle of one shard");
    if (n_shards == 0 || n_shards > kMaxShards) return fail(CLS_ERR_INVALID_ARGUMENT, "need 1 <= n_shards <= 8");
    uint64_t *seg[kMaxShards] = {nullptr};
    for (uint32_t o = 0; o < n_shards; ++o) seg[o] = (uint64_t *)d_send + (uint64_t)o * seg_cap;
    return route_hashes_impl(ix, rb, n_shards, seg_cap, seg, d_slot_win, counts_out, stream);
} CLS_ABI_CATCH

int cls_route_hashes_p2p(cls_index *ix, cls_resident_batch *rb, uint32_t n_shards, uint64_t seg_cap, void *const *d_segments,
                         void *d_slot_win, uint64_t *counts_out, void *stream) try {
    if (!ix || !rb || !d_segments || !d_slot_win || !counts_out) return fail(CLS_ERR_INVALID_ARGUMENT, "NULL argument");
    if (!ix->shards.empty()) return fail(CLS_ERR_INVALID_ARGUMENT, "a sharded handle routes internally: the routed calls take the handle of one shard");
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
    if (!ix->shards.empty()) return fail(CLS_ERR_INVALID_ARGUMENT, "a sharded handle routes internally: the routed calls take the handle of one shard");
    CU_TRY(cudaSetDevice(ix->device));
    cudaError_t e = launch_shard_probe(ix->dix, ix->shard, (const uint64_t *)d_hashes, n, d_replies, (cudaStream_t)stream);
    if (e != cudaSuccess) return fail(CLS_ERR_CUDA, std::string("probe kernel launch: ") + cudaGetErrorString(e));
    return CLS_OK;
} CLS_ABI_CATCH

int cls_place_routed(cls_index *ix, cls_resident_batch *rb, const void *d_replies, const void *d_slot_win,
                     uint32_t n_shards, uint64_t seg_cap, const cls_params *params, void *stream) try {
    if (!ix || !rb || !params || !d_replies || !d_slot_win) return fail(CLS_ERR_INVALID_ARGUMENT, "NULL argument");
    if (!ix->shards.empty()) return fail(CLS_ERR_INVALID_ARGUMENT, "a sharded handle routes internally: the routed calls take the handle of one shard");
    if (n_shards == 0 || n_shards > kMaxShards) return fail(CLS_ERR_INVALID_ARGUMENT, "need 1 <= n_shards <= 8");
    if (!rb->d_runs.p) return fail(CLS_ERR_INVALID_ARGUMENT, "cls_route_hashes has not run on this batch");
    CU_TRY(cudaSetDevice(ix->device));
    const PlaceParams pp = make_place_params(params);
    size_t want = 0;
    for (const LengthClass &c : rb->lay.classes) want = std::max(want, place_scratch_bytes(c.count, c.max_len, ix->dix.k_size, ix->dix.max_fanout));
    if (want > rb->d_scratch.cap) {
        if (rb->d_scratch.p) CU_TRY(cudaStreamSynchronize((cudaStream_t)stream));
        CU_TRY(rb->d_scratch.reserve(want));
    }
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

int cls_get_timing(const cls_index *ix, cls_timing *out) try {
    if (!ix || !out) return fail(CLS_ERR_INVALID_ARGUMENT, "NULL argument");
    std::lock_guard<std::mutex> lk(const_cast<cls_index *>(ix)->mu);
    *out = ix->timing;
    return CLS_OK;
} CLS_ABI_CATCH

int cls_debug_kmer_hashes(int device, uint32_t k_size, const uint8_t *bases, uint64_t len, uint64_t *out_hashes,
                          uint64_t cap, uint64_t *n_out) try {
    if (!n_out || (len && !bases) || k_size == 0) return fail(CLS_ERR_INVALID_ARGUMENT, "NULL argument or k == 0");
    *n_out = 0;
    if (len < k_size) return CLS_OK;  // kmers_map.rs:383-385
    if (len >= (1ull << 20)) return fail(CLS_ERR_UNSUPPORTED, "debug export is limited to 2^20 bases");
    CU_TRY(cudaSetDevice(device));
    const uint64_t n = 2 * (len - k_size + 1);
    std::vector<uint32_t> words((len + 15) / 16 + 2, 0);
    if (!pack_read(bases, (uint32_t)len, words.data())) return fail(CLS_ERR_INVALID_ARGUMENT, "non-ACGT byte in the sequence");
    DevBuf d_words, d_out;
    struct Free { DevBuf &a, &b; ~Free() { a.release(); b.release(); } } guard{d_words, d_out};
    CU_TRY(d_words.reserve(words.size() * 4));
    CU_TRY(d_out.reserve(n * 8));
    CU_TRY(cudaMemcpy(d_words.p, words.data(), words.size() * 4, cudaMemcpyHostToDevice));
    CU_TRY(launch_hash_only((const uint32_t *)d_words.p, (uint32_t)len, k_size, (uint64_t *)d_out.p, nullptr));
    CU_TRY(cudaDeviceSynchronize());
    std::vector<uint64_t> h(n);
    CU_TRY(cudaMemcpy(h.data(), d_out.p, n * 8, cudaMemcpyDeviceToHost));
    *n_out = n;
    if (out_hashes) std::memcpy(out_hashes, h.data(), std::min<uint64_t>(n, cap) * 8);
    return CLS_OK;
} CLS_ABI_CATCH

int cls_debug_node_counts(cls_index *ix, const uint8_t *bases, uint64_t len, const cls_params *params, cls_level_count *rows,
                          uint64_t cap, uint64_t *n_rows, cls_result *result) try {
    if (!ix || !params || !n_rows || (len && !bases) || (cap && !rows)) return fail(CLS_ERR_INVALID_ARGUMENT, "NULL argument");
    if (!ix->shards.empty()) return fail(CLS_ERR_INVALID_ARGUMENT, "this handle is sharded: no shard holds the whole table");
    if (!ix->replicas.empty()) ix = ix->replicas[0].get();   // a multi-device handle: resident batches live on its first device
    *n_rows = 0;
    if (ix->n_shards > 1) return fail(CLS_ERR_INVALID_ARGUMENT, "this handle holds one shard of the index");
    if (len < ix->dix.k_size || len >= (1ull << 20)) return fail(CLS_ERR_INVALID_ARGUMENT, "query shorter than k or longer than 2^20 bases");
    static_assert(sizeof(cls_level_count) == sizeof(TraceRow), "trace row layout");
    CU_TRY(cudaSetDevice(ix->device));
    std::vector<uint32_t> words((len + 15) / 16 + 8, 0);
    if (!pack_read(bases, (uint32_t)len, words.data())) return fail(CLS_ERR_INVALID_ARGUMENT, "non-ACGT byte in the sequence");
    const uint32_t cap_dev = (uint32_t)std::min<uint64_t>(std::max<uint64_t>(cap, 1), 1u << 22);
    DevBuf d_words, d_desc, d_res, d_rows, d_n;
    struct Free { DevBuf *b[5]; ~Free() { for (auto *x : b) x->release(); } } guard{{&d_words, &d_desc, &d_res, &d_rows, &d_n}};
    CU_TRY(d_words.reserve(words.size() * 4)); CU_TRY(d_desc.reserve(sizeof(ReadDesc))); CU_TRY(d_res.reserve(sizeof(ResultRec)));
    CU_TRY(d_rows.reserve((size_t)cap_dev * sizeof(TraceRow))); CU_TRY(d_n.reserve(4));
    const ReadDesc rd{0u, (uint32_t)len};
    CU_TRY(cudaMemcpy(d_words.p, words.data(), words.size() * 4, cudaMemcpyHostToDevice));
    CU_TRY(cudaMemcpy(d_desc.p, &rd, sizeof rd, cudaMemcpyHostToDevice));
    CU_TRY(cudaMemset(d_n.p, 0, 4));
    const PlaceGeom g = make_place_geom((uint32_t)len, ix->dix.k_size, ix->dix.max_fanout);
    cudaError_t e = launch_trace(ix->dix, make_place_params(params), (const uint32_t *)d_words.p, (const ReadDesc *)d_desc.p,
                                 (ResultRec *)d_res.p, g, ix->sm_count, nullptr, TraceBuf{(TraceRow *)d_rows.p, (uint32_t *)d_n.p, cap_dev});
    if (e != cudaSuccess) return fail(e == cudaErrorInvalidConfiguration ? CLS_ERR_UNSUPPORTED : CLS_ERR_CUDA, std::string("trace launch: ") + cudaGetErrorString(e));
    CU_TRY(cudaDeviceSynchronize());
    uint32_t n = 0;
    ResultRec rr;
    CU_TRY(cudaMemcpy(&n, d_n.p, 4, cudaMemcpyDeviceToHost));
    CU_TRY(cudaMemcpy(&rr, d_res.p, sizeof rr, cudaMemcpyDeviceToHost));
    *n_rows = n;
    const uint32_t take = (uint32_t)std::min<uint64_t>(std::min<uint32_t>(n, cap_dev), cap);
    if (take) {
        CU_TRY(cudaMemcpy(rows, d_rows.p, (size_t)take * sizeof(TraceRow), cudaMemcpyDeviceToHost));
        // rows arrive in no particular order within a level: sort by (level, child id) for the caller
        std::sort(rows, rows + take, [](const cls_level_count &a, const cls_level_count &b) {
            return a.level != b.level ? a.level < b.level : a.child_id < b.child_id;
        });
    }
    if (result) {
        if (result->status) result->status[0] = (uint8_t)rr.status;
        if (result->node_id) result->node_id[0] = rr.node_id;
        if (result->one) result->one[0] = rr.one;
        if (result->rest) result->rest[0] = rr.rest;
        if (result->n_query_kmers) result->n_query_kmers[0] = (uint32_t)(2 * (len - ix->dix.k_size + 1));
        if (result->n_matched) result->n_matched[0] = rr.n_matched;
        if (result->n_root_matched) result->n_root_matched[0] = rr.n_root_matched;
        if (result->iterations) result->iterations[0] = rr.iterations;
    }
    return CLS_OK;
} CLS_ABI_CATCH

int cls_debug_plan_batch(uint32_t k_size, const cls_batch *batch, uint8_t *pre_status, uint32_t *perm, uint32_t *word_off,
                         cls_plan_class *classes, uint32_t cap_classes, uint32_t *n_classes, uint32_t *n_device, uint64_t *n_words) try {
    if (!batch || !n_classes || !n_device || !n_words || k_size == 0) return fail(CLS_ERR_INVALID_ARGUMENT, "NULL argument or k == 0");
    PackedLayout lay;
    std::vector<uint32_t> woff;
    const int rc = plan_batch(batch, k_size, 0, lay, woff);
    if (rc != CLS_OK) return rc;
    *n_device = lay.n_device;
    *n_words = lay.n_words;
    *n_classes = (uint32_t)lay.classes.size();
    if (pre_status) std::memcpy(pre_status, lay.pre_status.data(), lay.pre_status.size());
    if (perm) std::memcpy(perm, lay.perm.data(), lay.perm.size() * 4);
    if (word_off) std::memcpy(word_off, woff.data(), woff.size() * 4);
    for (uint32_t c = 0; c < lay.classes.size() && c < cap_classes && classes; ++c)
        classes[c] = cls_plan_class{lay.classes[c].first, lay.classes[c].count, lay.classes[c].max_len};
    return CLS_OK;
} CLS_ABI_CATCH

int cls_debug_plan_fast(uint32_t k_size, const cls_batch *batch, uint64_t chunk_reads, uint32_t *word_off, uint32_t *lens,
                        uint64_t *src_off, uint32_t *max_len, uint64_t *n_planned) try {
    if (!batch || !n_planned || k_size == 0 || chunk_reads == 0) return fail(CLS_ERR_INVALID_ARGUMENT, "NULL argument, k == 0 or chunk_reads == 0");
    const uint64_t n = batch->n_queries;
    *n_planned = 0;
    if (max_len) *max_len = 0;
    if (n == 0) return CLS_OK;
    if (!batch->offsets || n >= 0xFFFFFFFFull) return fail(CLS_ERR_INVALID_ARGUMENT, "batch arrays are NULL or too long");
    PackedLayout lay;
    std::vector<uint32_t> woff((size_t)n + 1);
    std::vector<ReadDesc> descs(n);
    std::vector<uint64_t> src(n);
    lay.pre_status.resize(n); lay.lens.resize(n); lay.perm.resize(n);
    uint64_t words = 0, planned = 0;
    uint32_t mx = 0;
    const uint64_t base0 = batch->offsets[0];
    while (planned < n) {   // chunk by chunk, as place_batch_impl does
        const uint64_t end = std::min(n, planned + chunk_reads);
        if (!plan_reads_fast(batch, k_size, lay, woff, planned, end, words, mx, descs.data(), src.data(), base0)) break;
        planned = end;
    }
    *n_planned = planned;
    if (max_len) *max_len = mx;
    for (uint64_t i = 0; i < planned; ++i) {
        if (lay.perm[i] != i || lay.pre_status[i] != 0xFF || descs[i].word_off != woff[i] || descs[i].len != lay.lens[i])
            return fail(CLS_ERR_INVALID_ARGUMENT, "internal: the just-in-time plan is inconsistent");
    }
    if (word_off) std::memcpy(word_off, woff.data(), (size_t)(planned + (planned ? 1 : 0)) * 4);
    if (lens) std::memcpy(lens, lay.lens.data(), (size_t)planned * 4);
    if (src_off) std::memcpy(src_off, src.data(), (size_t)planned * 8);
    return CLS_OK;
} CLS_ABI_CATCH

int cls_debug_pack_read(const uint8_t *bases, uint64_t len, uint32_t *words_out, uint64_t cap_words, int portable) try {
    if ((len && !bases) || !words_out || len >= (1ull << 31) || cap_words < (len + 15) / 16)
        return fail(CLS_ERR_INVALID_ARGUMENT, "bad arguments");
    if (portable < 0 || portable > kPackAvx512) return fail(CLS_ERR_INVALID_ARGUMENT, "unknown packer variant");
    if (len == 0) return 1;
    const int r = pack_read_variant(portable, bases, (uint32_t)len, words_out);
    if (r < 0) return fail(CLS_ERR_UNSUPPORTED, "this CPU cannot run the requested packer variant");
    return r;
} CLS_ABI_CATCH

uint64_t cls_debug_host_murmur3_x64_128_h1(const uint8_t *data, uint64_t len, uint64_t seed) {
    return murmur3_x64_128_h1(data, len, seed);
}

}  // extern "C"
