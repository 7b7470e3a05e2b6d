// cls_place_batch on a single-device handle and on a multi-device one: planning, packing (host or device), the chunked
// three-stream pipeline, its workspaces, and the scatter of the 32-byte device result records into the caller's arrays.
// The planner and the packers also serve resident batches and the sharded handle.  All arithmetic of the placement runs
// in kernels; there is no CPU fallback here.
#include <cmath>
#include <thread>

#include "capi_internal.hpp"
#include "host_pack.hpp"

using namespace cls;

namespace cls {

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
                uint32_t *words, ReadDesc *descs, uint64_t first, uint64_t count) {
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

// Descriptors and source offsets (from `base0` on in the caller's bases) of the reads [first, first + count) of the device
// order, for packing on the device; returns how far into the bases those reads reach.
uint64_t fill_pack_descs(const cls_batch *batch, const PackedLayout &lay, uint64_t base0, uint64_t first, uint64_t count,
                         ReadDesc *descs, uint64_t *src) {
    std::atomic<uint64_t> need{0};
    parallel_for(count, 16384, [&](uint64_t a0, uint64_t b0) {
        uint64_t mx = 0;
        for (uint64_t j = first + a0; j < first + b0; ++j) {
            const uint64_t i = lay.perm[j];
            descs[j] = ReadDesc{lay.word_off[j], lay.lens[i]};
            src[j] = batch->offsets[i] - base0;
            mx = std::max(mx, batch->offsets[i + 1] - base0);
        }
        uint64_t cur = need.load();
        while (cur < mx && !need.compare_exchange_weak(cur, mx)) {}
    });
    return need.load();
}

// Reads of a batch planned just in time (place_batch_impl, `fast`): the optimistic plan of a batch of short reads - every
// read has k .. 162 bases (one geometry of the scan kernel), so the device order is the input order, nothing is decided
// on the host, and the layout of a chunk (word offsets, lengths) is written right before the chunk is enqueued instead of
// in a pass over the whole batch before the first copy starts (0.7 ms per million reads on sixteen threads, 2.7 ms on
// four: SCALE_r01's end-to-end curve).  Returns false - nothing written beyond `end` - when a read does not qualify;
// the caller then starts over with the general plan (plan_batch).
bool plan_reads_fast(const cls_batch *batch, uint32_t k, PackedLayout &lay, std::vector<uint32_t> &word_off, uint64_t first,
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

// The scratch buffer the placement of `classes` needs (the largest class's).
size_t scratch_for(const std::vector<LengthClass> &classes, const cls_index *ix) {
    size_t want = 0;
    for (const LengthClass &c : classes) want = std::max(want, place_scratch_bytes(c.count, c.max_len, ix->dix.k_size, ix->dix.max_fanout));
    return want;
}

// Growing the scratch buffer frees it: an earlier placement on `stream` may still use it, and is waited for first.
int grow_scratch(DevBuf &scratch, cudaStream_t stream, size_t bytes) {
    if (bytes > scratch.cap && scratch.p) CU_TRY(cudaStreamSynchronize(stream));
    CU_TRY(scratch.reserve(bytes));
    return CLS_OK;
}

int launch_classes(cls_index *ix, const PackedLayout &lay, const cls_params *params, const uint32_t *d_words,
                   const ReadDesc *d_descs, ResultRec *d_results, cudaStream_t stream, DevBuf &scratch, uint64_t *launches) {
    const PlaceParams pp = make_place_params(params);
    const int rc = grow_scratch(scratch, stream, scratch_for(lay.classes, ix));
    if (rc != CLS_OK) return rc;
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
void scatter_host_decided(const PackedLayout &lay, uint32_t k, cls_result *out, uint64_t first, uint64_t end) {
    if (end > lay.n_queries) end = lay.n_queries;
    if (first >= end) return;
    parallel_for(end - first, 65536, [&](uint64_t a0, uint64_t b0) {
        for (uint64_t i = first + a0; i < first + b0; ++i) {
            const uint64_t len = lay.lens[i];
            const uint8_t ps = lay.pre_status[i];
            if (out->n_query_kmers) out->n_query_kmers[i] = len >= k ? (uint32_t)(2 * (len - k + 1)) : 0u;
            if (ps != 0xFF) {
                if (out->status) out->status[i] = ps;
                zero_row(out, i);
            }
        }
    });
}

// Device result records [first, first + count) (device order) -> the caller's arrays (caller order).
// Queries demoted on the host while packing (invalid base) keep their host status.
void scatter_device_range(const PackedLayout &lay, const ResultRec *recs, cls_result *out, uint64_t first, uint64_t count,
                          const uint8_t *bad) {
    parallel_for(count, 65536, [&](uint64_t a, uint64_t b) {
        for (uint64_t j = first + a; j < first + b; ++j) {
            const uint64_t i = lay.perm[j];
            const ResultRec &r = recs[j];
            if (lay.pre_status[i] != 0xFF || (bad && bad[j])) {   // bad: flagged by the device packer
                if (out->status) out->status[i] = lay.pre_status[i] != 0xFF ? lay.pre_status[i] : (uint8_t)CLS_STATUS_ERR_INVALID_BASE;
                zero_row(out, i);
                continue;
            }
            write_row(out, i, r);
        }
    });
}

static Workspace *acquire_ws(cls_index *ix) {
    std::lock_guard<std::mutex> lk(ix->mu);
    for (auto &w : ix->pool)
        if (!w->in_use) { w->in_use = true; return w.get(); }
    auto w = std::make_unique<Workspace>();   // (nothing half-made is left behind)
    for (cudaStream_t *s : {&w->stream, &w->stream2, &w->stream3})
        if (cudaStreamCreateWithFlags(s, cudaStreamNonBlocking) != cudaSuccess) return nullptr;
    w->in_use = true;
    ix->pool.push_back(std::move(w));
    return ix->pool.back().get();
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
        std::lock_guard<std::mutex> lk(ix->mu);
        w->in_use = false;
    }
};


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
            const uint64_t need = fast ? batch->offsets[(uint64_t)c.first + c.count] - base0
                                       : fill_pack_descs(batch, lay, base0, c.first, c.count, h_descs, h_src);
            CU_TRY(cudaEventRecord(ev[0], st_in));
            CU_TRY(cudaMemsetAsync(d_bad + c.first, 0, c.count, st_in));
            // (just-in-time plan: the device order is the input order, a chunk's bases are one range - the ranges of
            // host-packed chunks are never sent)
            if (fast && uploaded < h_src[c.first]) uploaded = h_src[c.first];
            rc = upload_to(need);
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
        rc = grow_scratch(scratch, st_k, place_scratch_bytes(c.count, c.max_len, ix->dix.k_size, ix->dix.max_fanout));
        if (rc != CLS_OK) return rc;
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
std::vector<uint64_t> cut_by_bases(const cls_batch *batch, size_t nd) {
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
cls_result result_from(const cls_result *result, uint64_t a) {
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
        if (rcs[d] != CLS_OK) errs[d] = cls_last_error();   // thread-local: carry it to the caller's thread
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

}  // namespace cls

extern "C" int cls_place_batch(cls_index *ix, const cls_batch *batch, const cls_params *params, cls_result *result) try {
    if (!ix || !batch || !params || !result) return fail(CLS_ERR_INVALID_ARGUMENT, "NULL argument");
    if (ix->sharded) return ix->sharded->place_batch(ix, batch, params, result);
    if (!ix->replicas.empty()) return place_batch_multi(ix, batch, params, result);
    return place_batch_one(ix, batch, params, result);
} CLS_ABI_CATCH
