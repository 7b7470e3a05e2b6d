// The C ABI with the hash-sharded handle (cls_index_create_sharded, include/classeq_b200.h): capi.cu plus the routed
// pipeline behind one handle - route -> probe -> place inside one process, peer stores over NVLink, events across devices.
// One translation unit with capi.cu, whose planning, packing, buffers and scatter it shares; capi.cu reaches these calls
// only through the handle's ShardedCalls, so it still builds on its own against a runtime without peer access (the fake
// CUDA runtime of tests/test_capi_fake.py).  The library is built from this file.
#include <functional>

#include "capi.cu"

constexpr uint32_t kRoutedMaxLen = 161;
static const char *const kRoutedTooLong = "the routed path places reads of up to 161 bases (the one-warp-per-read geometry)";

// Reads per home and sub-batch: at config 5 (k = 35, 150 bp) 2^19 reads are 121.6 M windows, seg_cap = 17.5 M slots on eight
// shards and 3.1 GB of exchange buffers per GPU (inbox 8 bytes, reply 12, window 2 per slot).  CLS_SHARD_SUB_READS lowers it
// (tests: several sub-batches out of small batches).
static uint64_t shard_sub_reads() {
    static const uint64_t v = [] {
        const char *e = getenv("CLS_SHARD_SUB_READS");
        const long long x = e ? atoll(e) : 0;
        return x > 0 ? (uint64_t)x : (uint64_t)1 << 19;
    }();
    return v;
}

// Slots per (owner, sender) segment for `windows` k-mers at the busiest home: the expected share plus slack, in whole
// 128-byte lines of hashes (a multiple of 32 slots keeps the probe kernel's 384-byte reply rows aligned, DESIGN.md section 6).
static uint64_t seg_cap_for(uint64_t windows, uint32_t n_shards, bool exact) {
    const uint64_t c = exact ? windows : (uint64_t)((double)windows / n_shards * 1.15) + 65536;
    return (std::max<uint64_t>(c, 1) + 31) & ~(uint64_t)31;
}

// One home's reads of a sub-batch, packed on its device: the ranges [first, first + count) of its device order.
struct HomeWork {
    const uint32_t *words = nullptr;
    const ReadDesc *descs = nullptr;
    ResultRec *results = nullptr;
    uint2 *runs = nullptr;
    std::vector<LengthClass> ranges;
    uint64_t windows = 0;
};

static uint64_t windows_of(const PackedLayout &lay, const std::vector<LengthClass> &ranges, uint32_t k) {
    uint64_t w = 0;
    for (const LengthClass &c : ranges)
        for (uint32_t j = c.first; j < c.first + c.count; ++j) w += 2ull * (lay.lens[lay.perm[j]] - k + 1);
    return w;
}

// Leaves nothing of a failed call in flight on the lanes: the next call reuses (or grows, i.e. frees) their buffers.
struct LaneGuard {
    cls_index *front;
    bool clean = false;
    ~LaneGuard() {
        if (clean) return;
        for (auto &ln : front->lanes) {
            cudaSetDevice(ln->device);
            cudaStreamSynchronize(ln->stream);
        }
    }
};

// Enqueues route (every home) -> probe (every owner, every sender) -> place (every home) of one sub-batch on the lanes'
// streams, chained by events across devices: the host waits for nothing in between.  Ends with the copy of every home's
// route state (cursors, overflow flag) to the host.
static int enqueue_routed(cls_index *front, std::vector<HomeWork> &homes, const PlaceParams &pp, uint64_t seg_cap, cls_timing &tm) {
    const uint32_t n = (uint32_t)front->shards.size(), k = front->dix.k_size, fan = front->dix.max_fanout;
    if ((uint64_t)n * seg_cap >= 0xFFFFFFFFull) return fail(CLS_ERR_UNSUPPORTED, "exchange buffers beyond 2^32 entries: fewer reads per sub-batch");
    for (uint32_t s = 0; s < n; ++s) {   // (nothing of an earlier sub-batch is in flight: growing a buffer frees it)
        ShardLane &ln = *front->lanes[s];
        CU_TRY(cudaSetDevice(ln.device));
        CU_TRY(ln.inbox.reserve((size_t)n * seg_cap * 8));
        CU_TRY(ln.reply.reserve((size_t)n * seg_cap * kProbeReplyBytes));
        CU_TRY(ln.slot_win.reserve((size_t)n * seg_cap * 2));
        size_t want = 16;
        for (const LengthClass &c : homes[s].ranges) want = std::max(want, place_scratch_bytes(c.count, c.max_len, k, fan));
        CU_TRY(ln.d_scratch.reserve(want));
    }
    // 1. every home hashes its reads and stores every hash into its owner's inbox, segment `home` (a peer store)
    for (uint32_t h = 0; h < n; ++h) {
        ShardLane &ln = *front->lanes[h];
        CU_TRY(cudaSetDevice(ln.device));
        CU_TRY(cudaEventRecord(ln.t_begin, ln.stream));
        CU_TRY(cudaMemsetAsync(ln.state.p, 0, 128, ln.stream));
        uint64_t *seg[kMaxShards] = {nullptr};
        for (uint32_t o = 0; o < n; ++o) seg[o] = (uint64_t *)front->lanes[o]->inbox.p + (uint64_t)h * seg_cap;
        for (const LengthClass &c : homes[h].ranges) {
            const PlaceGeom g = make_place_geom(c.max_len, k, fan);
            const cudaError_t e = launch_route(k, homes[h].words, homes[h].descs, c.first, c.count, g, n, seg_cap, seg, (uint16_t *)ln.slot_win.p,
                                               homes[h].runs, (unsigned long long *)ln.state.p, (uint32_t *)((char *)ln.state.p + 64),
                                               front->shards[h]->sm_count, ln.stream);
            if (e == cudaErrorInvalidConfiguration) return fail(CLS_ERR_UNSUPPORTED, kRoutedTooLong);
            if (e != cudaSuccess) return fail(CLS_ERR_CUDA, std::string("route kernel launch: ") + cudaGetErrorString(e));
            tm.kernel_launches += 1;
        }
        CU_TRY(cudaEventRecord(ln.route_ev, ln.stream));
    }
    // 2. every owner answers every sender's segment straight into that sender's reply box, segment `owner`.  The senders in
    //    staggered order (owner, owner + 1, ...): in one order for all, every owner stored into one GPU at a time (DESIGN.md
    //    section 6).  A segment's count is the sender's cursor, read by the probe kernel itself.
    for (uint32_t o = 0; o < n; ++o) {
        ShardLane &ln = *front->lanes[o];
        CU_TRY(cudaSetDevice(ln.device));
        for (uint32_t j = 0; j < n; ++j) {
            const uint32_t h = (o + j) % n;
            const ShardLane &home = *front->lanes[h];
            CU_TRY(cudaStreamWaitEvent(ln.stream, home.route_ev, 0));
            const cudaError_t e = launch_shard_probe_counted(front->shards[o]->dix, o, (const uint64_t *)ln.inbox.p + (uint64_t)h * seg_cap, seg_cap,
                                                     (const unsigned long long *)home.state.p + o,
                                                     (char *)home.reply.p + (uint64_t)o * seg_cap * kProbeReplyBytes, front->shards[o]->sm_count, ln.stream);
            if (e != cudaSuccess) return fail(CLS_ERR_CUDA, std::string("probe kernel launch: ") + cudaGetErrorString(e));
            tm.kernel_launches += 1;
        }
        CU_TRY(cudaEventRecord(ln.probe_ev, ln.stream));
    }
    // 3. every home counts and descends once every owner has answered
    for (uint32_t h = 0; h < n; ++h) {
        ShardLane &ln = *front->lanes[h];
        CU_TRY(cudaSetDevice(ln.device));
        for (uint32_t o = 0; o < n; ++o) CU_TRY(cudaStreamWaitEvent(ln.stream, front->lanes[o]->probe_ev, 0));
        for (const LengthClass &c : homes[h].ranges) {
            const PlaceGeom g = make_place_geom(c.max_len, k, fan);
            const cudaError_t e = launch_place_routed(front->shards[h]->dix, pp, homes[h].words, homes[h].descs, c.first, c.count, homes[h].results, g, n,
                                                      seg_cap, homes[h].runs, (const uint16_t *)ln.slot_win.p, ln.reply.p, front->shards[h]->sm_count,
                                                      ln.stream, ln.d_scratch.p, ln.d_scratch.cap);
            if (e == cudaErrorInvalidConfiguration) return fail(CLS_ERR_UNSUPPORTED, kRoutedTooLong);
            if (e != cudaSuccess) return fail(CLS_ERR_CUDA, std::string("routed place kernel launch: ") + cudaGetErrorString(e));
            tm.kernel_launches += 1;
        }
        CU_TRY(cudaEventRecord(ln.t_end, ln.stream));
        CU_TRY(cudaMemcpyAsync(ln.h_state.p, ln.state.p, 128, cudaMemcpyDeviceToHost, ln.stream));
    }
    return CLS_OK;
}

// The one host wait of a sub-batch: every lane drained.  `overflow`: some segment exceeded seg_cap (the sub-batch runs again).
static int wait_lanes(cls_index *front, bool &overflow, cls_timing &tm) {
    overflow = false;
    float dev_ms = 0.f;
    for (auto &ln : front->lanes) {
        CU_TRY(cudaSetDevice(ln->device));
        CU_TRY(cudaStreamSynchronize(ln->stream));
        overflow |= ((const uint32_t *)ln->h_state.p)[16] != 0;
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, ln->t_begin, ln->t_end) == cudaSuccess) dev_ms = std::max(dev_ms, ms);
        (void)cudaGetLastError();
    }
    tm.kernel_ms += dev_ms;
    return CLS_OK;
}

// Runs one sub-batch to the end: routed stages, then (when a low-complexity read sent more windows to one owner than a
// segment holds) once more with seg_cap = the busiest home's windows - an exact bound, as a segment only ever receives
// its sender's windows; the results of the first run are overwritten.  `d2h` enqueues the copies of the results.
static int run_sub_batch(cls_index *front, std::vector<HomeWork> &homes, const PlaceParams &pp, cls_timing &tm, const std::function<int()> &d2h) {
    uint64_t max_windows = 0;
    for (const HomeWork &hw : homes) max_windows = std::max(max_windows, hw.windows);
    if (max_windows == 0) return CLS_OK;
    const uint32_t n = (uint32_t)front->shards.size();
    for (int attempt = 0; attempt < 2; ++attempt) {
        int rc = enqueue_routed(front, homes, pp, seg_cap_for(max_windows, n, attempt > 0), tm);
        if (rc == CLS_OK) rc = d2h();
        if (rc != CLS_OK) return rc;
        bool overflow = false;
        if ((rc = wait_lanes(front, overflow, tm)) != CLS_OK) return rc;
        if (!overflow) return CLS_OK;
    }
    return fail(CLS_ERR_OUT_OF_MEMORY, "internal: a segment overflowed at its exact bound");
}

static int place_batch_sharded(cls_index *front, const cls_batch *batch, const cls_params *params, cls_result *result) {
    const double t0 = now_ms();
    const uint64_t nq = batch->n_queries;
    if (nq && (!batch->offsets || (batch->offsets[nq] > batch->offsets[0] && !batch->bases))) return fail(CLS_ERR_INVALID_ARGUMENT, "batch arrays are NULL");
    if (nq >= 0xFFFFFFFFull) return fail(CLS_ERR_INVALID_ARGUMENT, "more than 2^32-1 queries in one batch");
    std::atomic<bool> bad_offsets{false}, too_long{false};   // decided before anything is enqueued
    parallel_for(nq, 1 << 16, [&](uint64_t a, uint64_t b) {
        for (uint64_t i = a; i < b; ++i) {
            const uint64_t o0 = batch->offsets[i], o1 = batch->offsets[i + 1];
            if (o1 < o0) bad_offsets = true;
            else if (o1 - o0 > kRoutedMaxLen) too_long = true;
        }
    });
    if (bad_offsets) return fail(CLS_ERR_INVALID_ARGUMENT, "batch offsets are not non-decreasing");
    if (too_long) return fail(CLS_ERR_UNSUPPORTED, kRoutedTooLong);
    std::lock_guard<std::mutex> lk(front->call_mu);
    LaneGuard guard{front};
    const uint32_t n = (uint32_t)front->shards.size(), k = front->dix.k_size;
    const PlaceParams pp = make_place_params(params);
    const std::vector<uint64_t> cut = cut_by_bases(batch, n);
    const uint64_t per = shard_sub_reads();
    uint64_t n_sub = 0;
    for (uint32_t h = 0; h < n; ++h) n_sub = std::max(n_sub, (cut[h + 1] - cut[h] + per - 1) / per);
    double host_share = 0.0;
    const bool dev_pack = resolve_pack_mode(n, false, host_share) != kPackOnHost;
    cls_timing tm{};
    std::vector<uint64_t> first(n);
    for (uint64_t sb = 0; sb < n_sub; ++sb) {
        const double tp = now_ms();
        std::vector<HomeWork> homes(n);
        // each home: plan, pack (host or device), copy up - the resident-batch layout, on the home's device
        for (uint32_t h = 0; h < n; ++h) {
            ShardLane &ln = *front->lanes[h];
            first[h] = std::min(cut[h] + sb * per, cut[h + 1]);
            const cls_batch part{std::min(per, cut[h + 1] - first[h]), batch->bases, batch->offsets + first[h]};
            PackedLayout &lay = ln.lay;
            int rc = plan_batch(&part, k, front->dix.max_fanout, lay, lay.word_off);
            if (rc != CLS_OK) return rc;
            if (!lay.n_device) continue;
            CU_TRY(cudaSetDevice(ln.device));
            const size_t words_b = (size_t)lay.n_words * 4, descs_b = (size_t)lay.n_device * sizeof(ReadDesc), res_b = (size_t)lay.n_device * sizeof(ResultRec);
            CU_TRY(ln.d_words.reserve(words_b + 16)); CU_TRY(ln.d_descs.reserve(descs_b)); CU_TRY(ln.d_results.reserve(res_b));
            CU_TRY(ln.runs.reserve((size_t)lay.n_device * 8 * sizeof(uint2)));
            CU_TRY(ln.h_descs.reserve(descs_b)); CU_TRY(ln.h_results.reserve(res_b));
            ReadDesc *h_descs = (ReadDesc *)ln.h_descs.p;
            ln.dev_pack = dev_pack;
            if (!dev_pack) {
                CU_TRY(ln.h_words.reserve(words_b + 16));
                pack_batch(&part, lay, lay.word_off, (uint32_t *)ln.h_words.p, h_descs);
                CU_TRY(cudaMemcpyAsync(ln.d_words.p, ln.h_words.p, words_b, cudaMemcpyHostToDevice, ln.stream));
                tm.h2d_bytes += words_b;
            } else {   // the ASCII of the part goes up as it is (from the caller's memory when it is pinned) and is packed there
                const uint64_t base0 = part.offsets[0], ascii_b = part.offsets[part.n_queries] - base0;
                CU_TRY(ln.d_ascii.reserve(ascii_b + 16)); CU_TRY(ln.d_src.reserve((size_t)lay.n_device * 8)); CU_TRY(ln.d_bad.reserve(lay.n_device));
                CU_TRY(ln.h_src.reserve((size_t)lay.n_device * 8)); CU_TRY(ln.h_bad.reserve(lay.n_device));
                uint64_t *h_src = (uint64_t *)ln.h_src.p;
                parallel_for(lay.n_device, 16384, [&](uint64_t a, uint64_t b) {
                    for (uint64_t j = a; j < b; ++j) {
                        const uint64_t i = lay.perm[j];
                        h_descs[j] = ReadDesc{lay.word_off[j], lay.lens[i]};
                        h_src[j] = part.offsets[i] - base0;
                    }
                });
                const uint8_t *src = batch->bases + base0;
                if (!is_pinned_host(src) || !is_pinned_host(src + ascii_b - 1)) {
                    CU_TRY(ln.h_ascii.reserve(ascii_b));
                    uint8_t *dst = (uint8_t *)ln.h_ascii.p;
                    parallel_for(ascii_b, (uint64_t)1 << 20, [&](uint64_t a, uint64_t b) { memcpy(dst + a, src + a, b - a); });
                    src = dst;
                }
                CU_TRY(cudaMemcpyAsync(ln.d_ascii.p, src, ascii_b, cudaMemcpyHostToDevice, ln.stream));
                CU_TRY(cudaMemcpyAsync(ln.d_src.p, h_src, (size_t)lay.n_device * 8, cudaMemcpyHostToDevice, ln.stream));
                CU_TRY(cudaMemsetAsync(ln.d_bad.p, 0, lay.n_device, ln.stream));
                tm.h2d_bytes += ascii_b + (uint64_t)lay.n_device * 8;
            }
            CU_TRY(cudaMemcpyAsync(ln.d_descs.p, h_descs, descs_b, cudaMemcpyHostToDevice, ln.stream));
            tm.h2d_bytes += descs_b;
            if (dev_pack) {
                const cudaError_t e = launch_ascii_pack((const uint8_t *)ln.d_ascii.p, (const uint64_t *)ln.d_src.p, (const ReadDesc *)ln.d_descs.p, 0,
                                                        lay.n_device, lay.classes[0].max_len, (uint32_t *)ln.d_words.p, (uint8_t *)ln.d_bad.p, ln.stream);
                if (e != cudaSuccess) return fail(CLS_ERR_CUDA, std::string("pack kernel launch: ") + cudaGetErrorString(e));
                tm.kernel_launches += 1;
            }
            HomeWork &hw = homes[h];
            hw.words = (const uint32_t *)ln.d_words.p; hw.descs = (const ReadDesc *)ln.d_descs.p; hw.results = (ResultRec *)ln.d_results.p;
            hw.runs = (uint2 *)ln.runs.p; hw.ranges = lay.classes; hw.windows = windows_of(lay, lay.classes, k);
        }
        tm.pack_ms += now_ms() - tp;
        int rc = run_sub_batch(front, homes, pp, tm, [&]() -> int {
            for (uint32_t h = 0; h < n; ++h) {
                ShardLane &ln = *front->lanes[h];
                const uint32_t nd = ln.lay.n_device;
                if (!nd) continue;
                CU_TRY(cudaSetDevice(ln.device));
                CU_TRY(cudaMemcpyAsync(ln.h_results.p, ln.d_results.p, (size_t)nd * sizeof(ResultRec), cudaMemcpyDeviceToHost, ln.stream));
                tm.d2h_bytes += (uint64_t)nd * sizeof(ResultRec);
                if (ln.dev_pack) {
                    CU_TRY(cudaMemcpyAsync(ln.h_bad.p, ln.d_bad.p, nd, cudaMemcpyDeviceToHost, ln.stream));
                    tm.d2h_bytes += nd;
                }
            }
            return CLS_OK;
        });
        if (rc != CLS_OK) return rc;
        for (uint32_t h = 0; h < n; ++h) {
            ShardLane &ln = *front->lanes[h];
            cls_result r = result_from(result, first[h]);
            scatter_host_decided(ln.lay, k, &r);
            if (ln.lay.n_device)
                scatter_device_range(ln.lay, (const ResultRec *)ln.h_results.p, &r, 0, ln.lay.n_device, ln.dev_pack ? (const uint8_t *)ln.h_bad.p : nullptr);
        }
    }
    tm.total_ms = now_ms() - t0;
    tm.pack_on_device = dev_pack ? 1u : 0u;
    { std::lock_guard<std::mutex> lk2(front->mu); front->timing = tm; }
    guard.clean = true;
    return CLS_OK;
}

// A resident batch on the first shard's device, routed from there to every owner in sub-batches of its device order.
// Waits for the placement (the overflow check needs the host).
static int place_resident_sharded(cls_index *front, cls_resident_batch *rb, const cls_params *params, cudaStream_t stream) {
    const double t0 = now_ms();
    if (rb->device != front->device) return fail(CLS_ERR_INVALID_ARGUMENT, "resident batch lives on another device");
    for (const LengthClass &c : rb->lay.classes)
        if (c.max_len > kRoutedMaxLen) return fail(CLS_ERR_UNSUPPORTED, kRoutedTooLong);
    std::lock_guard<std::mutex> lk(front->call_mu);
    LaneGuard guard{front};
    const uint32_t n = (uint32_t)front->shards.size(), k = front->dix.k_size;
    const PlaceParams pp = make_place_params(params);
    ShardLane &home = *front->lanes[0];
    CU_TRY(cudaSetDevice(home.device));
    CU_TRY(rb->d_runs.reserve((size_t)rb->lay.n_device * 8 * sizeof(uint2) + 64));
    // what the caller enqueued on its stream before (the upload, an earlier placement) comes first
    CU_TRY(cudaEventRecord(home.t_begin, stream));
    CU_TRY(cudaStreamWaitEvent(home.stream, home.t_begin, 0));
    cls_timing tm{};
    const uint64_t per = shard_sub_reads();
    std::vector<HomeWork> homes(n);
    HomeWork &hw = homes[0];
    hw.words = (const uint32_t *)rb->d_words.p; hw.descs = (const ReadDesc *)rb->d_descs.p; hw.results = (ResultRec *)rb->d_results.p;
    hw.runs = (uint2 *)rb->d_runs.p;
    auto flush = [&]() -> int {
        hw.windows = windows_of(rb->lay, hw.ranges, k);
        const int rc = run_sub_batch(front, homes, pp, tm, [] { return (int)CLS_OK; });
        hw.ranges.clear();
        return rc;
    };
    uint64_t filled = 0;
    for (const LengthClass &c : rb->lay.classes)
        for (uint32_t a = 0; a < c.count;) {
            const uint32_t take = (uint32_t)std::min<uint64_t>(per - filled, c.count - a);
            hw.ranges.push_back(LengthClass{c.first + a, take, c.max_len});
            a += take;
            if ((filled += take) == per) {
                filled = 0;
                const int rc = flush();
                if (rc != CLS_OK) return rc;
            }
        }
    if (!hw.ranges.empty()) {
        const int rc = flush();
        if (rc != CLS_OK) return rc;
    }
    tm.total_ms = now_ms() - t0;
    { std::lock_guard<std::mutex> lk2(front->mu); front->timing = tm; }
    guard.clean = true;
    return CLS_OK;
}

static const cls_index::ShardedCalls kShardedCalls{place_batch_sharded, place_resident_sharded};

extern "C" {

int cls_index_create_sharded(const cls_model_view *model, uint32_t n_shards, const int *devices, cls_index **out) try {
    if (!out) return fail(CLS_ERR_INVALID_ARGUMENT, "out is NULL");
    *out = nullptr;
    if (n_shards == 0 || n_shards > kMaxShards || !devices) return fail(CLS_ERR_INVALID_ARGUMENT, "need 1 <= n_shards <= 8 and a device list");
    // every shard stores into every other shard's memory: peer access between every pair of distinct devices, or nothing
    for (uint32_t a = 0; a < n_shards; ++a)
        for (uint32_t b = 0; b < n_shards; ++b) {
            if (devices[a] == devices[b]) continue;
            int can = 0;
            CU_TRY(cudaDeviceCanAccessPeer(&can, devices[a], devices[b]));
            if (!can) return fail(CLS_ERR_UNSUPPORTED, "devices " + std::to_string(devices[a]) + " and " + std::to_string(devices[b]) +
                                                           " cannot access each other's memory (peer access): a sharded index needs it");
            CU_TRY(cudaSetDevice(devices[a]));
            const cudaError_t e = cudaDeviceEnablePeerAccess(devices[b], 0);
            if (e == cudaErrorPeerAccessAlreadyEnabled) (void)cudaGetLastError();
            else if (e != cudaSuccess) return fail(CLS_ERR_CUDA, std::string("cudaDeviceEnablePeerAccess: ") + cudaGetErrorString(e));
        }
    auto front = std::make_unique<cls_index>();
    for (uint32_t s = 0; s < n_shards; ++s) {
        HostIndex h;
        int rc = build_index_host(model, s, n_shards, h);
        if (rc != CLS_OK) return rc;
        std::unique_ptr<cls_index> sh;
        if ((rc = upload_index(h, devices[s], s, n_shards, sh)) != CLS_OK) return rc;
        front->shards.push_back(std::move(sh));
        front->lanes.push_back(std::make_unique<ShardLane>());
        ShardLane &ln = *front->lanes.back();
        ln.device = devices[s];
        CU_TRY(cudaStreamCreateWithFlags(&ln.stream, cudaStreamNonBlocking));
        CU_TRY(cudaEventCreateWithFlags(&ln.route_ev, cudaEventDisableTiming));
        CU_TRY(cudaEventCreateWithFlags(&ln.probe_ev, cudaEventDisableTiming));
        CU_TRY(cudaEventCreate(&ln.t_begin));
        CU_TRY(cudaEventCreate(&ln.t_end));
        CU_TRY(ln.state.reserve(128));
        CU_TRY(ln.h_state.reserve(128));
    }
    const cls_index &s0 = *front->shards[0];
    front->device = s0.device;
    front->sm_count = s0.sm_count;
    front->dix = s0.dix;
    front->info = s0.info;
    front->info.n_entries = front->info.n_buckets = front->info.table_bytes = 0;
    for (const auto &s : front->shards) {
        front->info.n_entries += s->info.n_entries;
        front->info.n_buckets += s->info.n_buckets;
        front->info.table_bytes += s->info.table_bytes;
    }
    front->info.n_devices = n_shards;
    front->sharded = &kShardedCalls;
    *out = front.release();
    return CLS_OK;
} CLS_ABI_CATCH

}  // extern "C"
