// C ABI of the placement path (include/classeq_b200.h): errors, version, parameters, creating and describing index
// handles, timing, the packing mode and the debug exports.  The placement calls are in place_batch.cpp, resident.cpp,
// routed.cpp and capi_sharded.cpp; there is no CPU fallback anywhere in them.
#include <thread>

#include "capi_internal.hpp"
#include "host_pack.hpp"
#include "murmur3_host.hpp"

using namespace cls;

namespace cls {

static thread_local std::string g_last_error;

int set_last_error(int code, const std::string &msg) {
    g_last_error = msg;
    return code;
}

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

// The host-built index `h` on one device.
int upload_index(const HostIndex &h, int device, uint32_t shard, uint32_t n_shards, std::unique_ptr<cls_index> &res) {
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
    CU_TRY(up(ix->tables.table, h.table.data(), h.table.size() * sizeof(Slot)));
    CU_TRY(up(ix->tables.arena, h.arena.data(), h.arena.size() * sizeof(SetWord)));
    CU_TRY(up(ix->tables.qnodes, h.qnodes.data(), h.qnodes.size() * sizeof(QNode)));
    CU_TRY(up(ix->tables.qchild, h.q_child_list.data(), h.q_child_list.size() * sizeof(uint32_t)));
    CU_TRY(up(ix->tables.qid, h.q_node_id.data(), h.q_node_id.size() * sizeof(uint64_t)));
    CU_TRY(up(ix->tables.terms, h.terms.data(), h.terms.size() * sizeof(uint32_t)));
    CU_TRY(up(ix->tables.qinfo, h.qinfo.data(), h.qinfo.size() * sizeof(QInfo)));
    CU_TRY(up(ix->tables.lca, h.lca_table.data(), h.lca_table.size() * sizeof(uint64_t)));
    ix->dix.table = (const Slot *)ix->tables.table.p;
    ix->dix.bucket_mask = h.n_buckets - 1;
    ix->dix.arena = (const SetWord *)ix->tables.arena.p;
    ix->dix.qnodes = (const QNode *)ix->tables.qnodes.p;
    ix->dix.q_child_list = (const uint32_t *)ix->tables.qchild.p;
    ix->dix.q_node_id = (const uint64_t *)ix->tables.qid.p;
    ix->dix.terms = (const uint32_t *)ix->tables.terms.p;
    ix->dix.qinfo = (const QInfo *)ix->tables.qinfo.p;
    ix->dix.lca_table = (const uint64_t *)ix->tables.lca.p;
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

int build_index_host(const cls_model_view *model, uint32_t shard, uint32_t n_shards, HostIndex &h) {
    std::string err;
    int rc = build_host_index(model, h, err, shard, n_shards);
    if (rc != CLS_OK) return fail(rc, err);
    if (h.n_buckets > (1ull << (n_shards > 1 ? 28 : 30))) return fail(CLS_ERR_UNSUPPORTED, "k-mer table too large (2^30 buckets, 2^28 per shard)");
    return CLS_OK;
}

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
PackMode resolve_pack_mode(size_t n_devices_of_handle, bool fast_plan, double &host_share) {
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

bool is_pinned_host(const void *p) {
    cudaPointerAttributes a{};
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { (void)cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost;
}

}  // namespace cls

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

int cls_set_pack_mode(int mode) {
    if (mode < 0 || mode > 3) return fail(CLS_ERR_INVALID_ARGUMENT, "pack mode must be 0 (automatic), 1 (host), 2 (device) or 3 (mixed)");
    const int prev = g_pack_mode.exchange(mode);
    return prev < 0 ? 0 : prev;
}

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
    ix = resident_home(ix);
    *n_rows = 0;
    if (ix->n_shards > 1) return fail(CLS_ERR_INVALID_ARGUMENT, "this handle holds one shard of the index");
    if (len < ix->dix.k_size || len >= (1ull << 20)) return fail(CLS_ERR_INVALID_ARGUMENT, "query shorter than k or longer than 2^20 bases");
    static_assert(sizeof(cls_level_count) == sizeof(TraceRow), "trace row layout");
    CU_TRY(cudaSetDevice(ix->device));
    std::vector<uint32_t> words((len + 15) / 16 + 8, 0);
    if (!pack_read(bases, (uint32_t)len, words.data())) return fail(CLS_ERR_INVALID_ARGUMENT, "non-ACGT byte in the sequence");
    const uint32_t cap_dev = (uint32_t)std::min<uint64_t>(std::max<uint64_t>(cap, 1), 1u << 22);
    DevBuf d_words, d_desc, d_res, d_rows, d_n;
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
        write_row(result, 0, rr);
        if (result->n_query_kmers) result->n_query_kmers[0] = (uint32_t)(2 * (len - ix->dix.k_size + 1));
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
