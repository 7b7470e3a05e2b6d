// TEST INFRASTRUCTURE.  The sharded handle (cls_index_create_sharded, classeq2_b200/csrc/capi_sharded.cu) end to end WITHOUT a GPU:
// the library's host side against the fake CUDA runtime (tests/native/fakecuda/), the three routed launches restated on the
// host (tests/native/fake_routed_kernels.cpp: route with the oracle's hash, probe over the shard's uploaded table, place_routed
// checking every reply against a direct probe of the owner shard before the oracle places the read).  Results must equal
// the oracle's on the caller's ASCII batch for 1, 3 and 8 shards over one to three devices: several sub-batches, host and
// device packing, a segment that overflows (the sub-batch runs again), the resident path and the FASTA ingest, concurrent
// callers, refused calls, failing allocations and failing CUDA calls.  Built with AddressSanitizer + UBSan and with
// ThreadSanitizer (FAKE_CUDA_ASYNC=1: every stream a worker thread) by tests/test_sharded_handle.py.
#include <atomic>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include <cuda_runtime.h>

#include "../../include/classeq_b200.h"

namespace fakek {
extern const void *oracle_model;
extern std::atomic<uint64_t> async_errors;
}  // namespace fakek
extern "C" {
void *orc_model_create(const void *view);
void orc_model_destroy(void *);
uint64_t orc_kmer_hashes(const uint8_t *bases, uint64_t len, uint32_t k, uint64_t *out, uint64_t cap);
void orc_place_batch(const void *model, const uint8_t *bases, const uint64_t *offsets, uint64_t n, int32_t max_iterations,
                     double min_match_coverage, uint32_t remove_intersection, int n_threads, uint8_t *status, uint64_t *node_id, int32_t *one,
                     int32_t *rest, uint32_t *n_query_kmers, uint32_t *n_matched, uint32_t *n_root_matched, uint32_t *iterations);
}

static uint64_t rng_state = 0x9E3779B97F4A7C15ull;
static uint64_t rnd() { rng_state ^= rng_state << 13; rng_state ^= rng_state >> 7; rng_state ^= rng_state << 17; return rng_state; }

struct Results {
    std::vector<uint8_t> status; std::vector<uint64_t> node; std::vector<int32_t> one, rest; std::vector<uint32_t> nq, nm, nr, it;
    explicit Results(uint64_t n) : status(n, 0xEE), node(n, ~0ull), one(n, -7), rest(n, -7), nq(n, 77), nm(n, 77), nr(n, 77), it(n, 77) {}
    cls_result view() { return cls_result{status.data(), node.data(), one.data(), rest.data(), nq.data(), nm.data(), nr.data(), it.data()}; }
    bool operator==(const Results &o) const { return status == o.status && node == o.node && one == o.one && rest == o.rest && nq == o.nq && nm == o.nm && nr == o.nr && it == o.it; }
};

struct Batch {
    std::vector<uint8_t> bases;
    std::vector<uint64_t> offsets{0};
    uint64_t n() const { return offsets.size() - 1; }
    cls_batch view(const uint8_t *b = nullptr) const { return cls_batch{n(), b ? b : bases.data(), offsets.data()}; }
    void add(const std::string &r) { bases.insert(bases.end(), r.begin(), r.end()); offsets.push_back(bases.size()); }
};

static std::atomic<long> g_bad{0}, g_reads{0};
#define EXPECT(c) do { if (!(c)) { ++g_bad; if (g_bad < 20) fprintf(stderr, "line %d: %s\n", __LINE__, #c); } } while (0)

static void compare(const Batch &b, Results &got, const void *orc, const cls_params &p, const char *what) {
    const uint64_t n = b.n();
    Results want(n);
    if (n) orc_place_batch(orc, b.bases.data(), b.offsets.data(), n, p.max_iterations, p.min_match_coverage, p.remove_intersection, 2,
                           want.status.data(), want.node.data(), want.one.data(), want.rest.data(), want.nq.data(), want.nm.data(),
                           want.nr.data(), want.it.data());
    long bad = 0;
    for (uint64_t i = 0; i < n; ++i) {
        bool invalid = false;
        for (uint64_t j = b.offsets[i]; j < b.offsets[i + 1]; ++j) { const uint8_t c = b.bases[j] & 0xDF; invalid |= !(c == 'A' || c == 'C' || c == 'G' || c == 'T'); }
        const uint64_t len = b.offsets[i + 1] - b.offsets[i];
        if (invalid && len >= 35) {
            bad += !(got.status[i] == CLS_STATUS_ERR_INVALID_BASE && got.node[i] == 0 && got.nm[i] == 0 && got.nq[i] == 2 * (len - 34));
            continue;
        }
        bad += !(got.status[i] == want.status[i] && got.node[i] == want.node[i] && got.one[i] == want.one[i] && got.rest[i] == want.rest[i] &&
                 got.nq[i] == want.nq[i] && got.nm[i] == want.nm[i] && got.nr[i] == want.nr[i] && got.it[i] == want.it[i]);
    }
    if (bad) fprintf(stderr, "%s: %ld of %llu queries differ\n", what, bad, (unsigned long long)n);
    g_bad += bad;
    g_reads += (long)n;
}

static uint32_t owner_of(uint64_t h, uint32_t n) { return (uint32_t)(h >> 61) % n; }

int main(int argc, char **argv) {
    const bool threads_only = argc > 1 && !strcmp(argv[1], "threads");   // the ThreadSanitizer build: fewer scenarios
    setenv("CLS_HOST_THREADS", "4", 0);
    setenv("CLS_SHARD_SUB_READS", "1500", 1);   // several sub-batches out of a few thousand reads
    // ---- a model: random binary tree over 24 tips, sequences evolved along it, k = 35, m = 4 ---------------------------------
    const uint32_t n_tips = 24;
    std::vector<uint64_t> node_id, child_off{0}, child_idx, tip_node;
    std::vector<uint8_t> kind;
    std::vector<std::string> seq_of_node;
    {
        std::vector<std::vector<uint64_t>> kids;
        std::vector<uint32_t> tips_below;
        auto add = [&](uint8_t k, const std::string &s, uint32_t t) { node_id.push_back(node_id.size() * 3 + 1); kind.push_back(k); seq_of_node.push_back(s); kids.emplace_back(); tips_below.push_back(t); return node_id.size() - 1; };
        std::string root_seq;
        for (int i = 0; i < 600; ++i) root_seq += "ACGT"[rnd() & 3];
        add(CLS_KIND_ROOT, root_seq, n_tips);
        for (uint64_t i = 0; i < node_id.size(); ++i) {
            if (tips_below[i] < 2) continue;
            const uint32_t left = 1 + (uint32_t)(rnd() % (tips_below[i] - 1));
            for (uint32_t part : {left, tips_below[i] - left}) {
                std::string s = seq_of_node[i];
                for (auto &c : s) if (rnd() % 40 == 0) c = "ACGT"[rnd() & 3];
                const uint64_t c = add(part == 1 ? CLS_KIND_LEAF : CLS_KIND_NODE, s, part);   // (grows `kids`)
                kids[i].push_back(c);
            }
        }
        for (uint64_t i = 0; i < node_id.size(); ++i) {
            for (uint64_t c : kids[i]) child_idx.push_back(c);
            child_off.push_back(child_idx.size());
            if (kind[i] == CLS_KIND_LEAF) tip_node.push_back(i);
        }
    }
    Batch refs;
    for (uint64_t t : tip_node) refs.add(seq_of_node[t]);
    cls_model_view tree{};
    tree.k_size = 35; tree.m_size = 4;
    tree.n_nodes = node_id.size(); tree.node_id = node_id.data(); tree.node_kind = kind.data(); tree.child_off = child_off.data(); tree.child_idx = child_idx.data();
    cls_built_model *bm = nullptr;
    if (cls_model_build(&tree, tip_node.size(), tip_node.data(), refs.bases.data(), refs.offsets.data(), &bm) != CLS_OK) { printf("model build failed\n"); return 1; }
    cls_model_view model{};
    cls_built_model_view(bm, &tree, &model);
    void *orc = orc_model_create(&model);
    fakek::oracle_model = orc;
    cls_params params;
    cls_params_default(&params);

    // reads of lo..hi bases from the tips (some unrelated, some with an invalid base when junk_every)
    auto make_reads = [&](uint64_t n, uint32_t lo, uint32_t hi, int junk_every) {
        Batch b;
        for (uint64_t i = 0; i < n; ++i) {
            const std::string &s = seq_of_node[tip_node[rnd() % tip_node.size()]];
            const uint32_t len = lo + (uint32_t)(rnd() % (hi - lo + 1));
            std::string r = s.substr(rnd() % (s.size() - len + 1), len);
            if (rnd() % 20 == 0) for (auto &c : r) c = "ACGT"[rnd() & 3];
            for (auto &c : r) if (rnd() % 100 == 0) c = "ACGT"[rnd() & 3];
            if (rnd() % 2) for (auto &c : r) if (rnd() % 7 == 0) c = (char)(c | 0x20);
            if (junk_every && i % junk_every == 3 && !r.empty()) r[rnd() % r.size()] = "NnX-"[rnd() % 4];
            b.add(r);
        }
        if (b.bases.empty()) b.bases.push_back('A');
        return b;
    };
    auto place = [&](cls_index *ix, const Batch &b, const cls_params &p, const char *what, const uint8_t *pinned = nullptr) {
        Results r(b.n());
        cls_result rv = r.view();
        const cls_batch bv = b.view(pinned);
        const int rc = cls_place_batch(ix, &bv, &p, &rv);
        EXPECT(rc == CLS_OK);
        if (rc != CLS_OK) fprintf(stderr, "%s: %s\n", what, cls_last_error());
        compare(b, r, orc, p, what);
    };

    cls_index *flat = nullptr;
    if (cls_index_create(&model, 0, &flat) != CLS_OK) { printf("index: %s\n", cls_last_error()); return 1; }
    cls_index_info flat_info{};
    cls_index_get_info(flat, &flat_info);

    // ---- 1. 1, 3 and 8 shards over one to three devices: ragged lengths (below k up to 161), host and device packing --------
    const std::vector<std::vector<int>> layouts = {{0}, {0, 1, 2}, {0, 0, 1}, {0, 1, 2, 0, 1, 2, 0, 1}};
    for (const auto &devs : layouts) {
        if (threads_only && devs.size() != 3) continue;
        cls_index *ix = nullptr;
        EXPECT(cls_index_create_sharded(&model, (uint32_t)devs.size(), devs.data(), &ix) == CLS_OK && ix);
        if (!ix) continue;
        cls_index_info info{};
        EXPECT(cls_index_get_info(ix, &info) == CLS_OK && info.n_devices == devs.size() && info.device == devs[0] &&
               info.n_entries == flat_info.n_entries && info.n_distinct_sets == flat_info.n_distinct_sets);
        for (int mode = 1; mode <= 2; ++mode) {
            cls_set_pack_mode(mode);
            const Batch b = make_reads(threads_only ? 3000 : 5000, 20, 161, 13);   // 5 000 reads on 3 homes: two sub-batches each
            cls_params p = params;
            p.remove_intersection = mode == 2;
            place(ix, b, p, "ragged");
            if (mode == 2 && !threads_only) {   // the bases in pinned memory: copied from there
                void *pin = nullptr;
                cudaHostAlloc(&pin, b.bases.size(), cudaHostAllocDefault);
                memcpy(pin, b.bases.data(), b.bases.size());
                place(ix, b, params, "ragged, pinned", static_cast<const uint8_t *>(pin));
                cudaFreeHost(pin);
            }
            cls_timing tm{};
            EXPECT(cls_get_timing(ix, &tm) == CLS_OK && tm.kernel_launches >= 3 && tm.pack_on_device == (mode == 2 ? 1u : 0u));
        }
        cls_set_pack_mode(0);
        {   // empty batch, only reads shorter than k
            Batch none;
            none.bases.push_back('A');
            place(ix, none, params, "empty");
            place(ix, make_reads(200, 1, 34, 0), params, "too short");
        }
        // ---- 2. resident batch on the first shard's device, routed to every owner --------------------------------------------
        {
            const Batch b = make_reads(2500, 30, 161, 0);
            const cls_batch bv = b.view();
            cls_resident_batch *rb = nullptr;
            EXPECT(cls_batch_upload(ix, &bv, &rb) == CLS_OK && rb);
            if (rb) {
                cudaStream_t user = nullptr;
                cudaSetDevice(devs[0]);
                cudaStreamCreateWithFlags(&user, cudaStreamNonBlocking);
                EXPECT(cls_place_resident(ix, rb, &params, user) == CLS_OK);
                Results r(b.n());
                cls_result rv = r.view();
                EXPECT(cls_resident_fetch(ix, rb, user, &rv) == CLS_OK);
                compare(b, r, orc, params, "resident");
                cudaStreamDestroy(user);
                cls_resident_destroy(rb);
            }
        }
        cls_index_destroy(ix);
    }
    // ---- 3. a segment overflows: low-complexity reads send every window to one owner; the sub-batch runs again --------------
    {
        // a homopolymer whose forward and reverse-complement windows share an owner, for some shard count
        uint32_t n_sh = 0;
        char base = 0;
        for (uint32_t n = 2; n <= 8 && !n_sh; ++n)
            for (char c : {'A', 'C'}) {
                const std::string r(150, c);
                std::vector<uint64_t> h(232);
                orc_kmer_hashes(reinterpret_cast<const uint8_t *>(r.data()), r.size(), 35, h.data(), h.size());
                bool one = true;
                for (uint64_t x : h) one &= owner_of(x, n) == owner_of(h[0], n);
                if (one && !n_sh) { n_sh = n; base = c; }
            }
        EXPECT(n_sh != 0);
        if (n_sh) {
            // every home gets 1 200 such reads: 278 400 windows to one owner, the first seg_cap holds 278 400 / n * 1.15 + 65 536
            const uint64_t per_home = 1200, windows = per_home * 232;
            EXPECT(windows > (uint64_t)(windows / (double)n_sh * 1.15) + 65536 + 32);
            Batch b;
            const Batch normal = make_reads(n_sh * 300, 100, 150, 0);
            for (uint64_t i = 0, j = 0; i < n_sh * per_home; ++i) {
                b.add(std::string(150, base));
                if (i % 4 == 0 && j < normal.n()) { b.add(std::string(normal.bases.begin() + (long)normal.offsets[j], normal.bases.begin() + (long)normal.offsets[j + 1])); ++j; }
            }
            std::vector<int> devs(n_sh);
            for (uint32_t s = 0; s < n_sh; ++s) devs[s] = (int)(s % 3);
            cls_index *ix = nullptr;
            EXPECT(cls_index_create_sharded(&model, n_sh, devs.data(), &ix) == CLS_OK);
            if (ix) {
                for (int mode = 1; mode <= 2; ++mode) {
                    if (threads_only && mode == 1) continue;
                    cls_set_pack_mode(mode);
                    place(ix, b, params, "overflow");
                }
                cls_set_pack_mode(0);
                cls_index_destroy(ix);
            }
        }
    }
    // ---- 4. concurrent callers on one handle; the FASTA ingest on the handle --------------------------------------------------
    {
        const int devs[3] = {0, 1, 2};
        cls_index *ix = nullptr;
        EXPECT(cls_index_create_sharded(&model, 3, devs, &ix) == CLS_OK);
        std::vector<Batch> bs;
        for (int t = 0; t < 4; ++t) bs.push_back(make_reads(1200, 35, 161, 0));
        std::vector<std::thread> th;
        for (int t = 0; t < 4; ++t) th.emplace_back([&, t] { for (int rep = 0; rep < 2; ++rep) place(ix, bs[t], params, "concurrent"); });
        for (auto &t : th) t.join();
        if (!threads_only) {
            std::string text;
            for (int i = 0; i < 300; ++i) {
                const std::string &s = seq_of_node[tip_node[rnd() % tip_node.size()]];
                const uint32_t len = 10 + (uint32_t)(rnd() % 150);
                text += ">q" + std::to_string(i) + "\n" + s.substr(rnd() % (s.size() - len), len) + "\n";
            }
            cls_resident_batch *rb = nullptr;
            cls_fasta_records dr{};
            EXPECT(cls_fasta_upload(ix, reinterpret_cast<const uint8_t *>(text.data()), text.size(), &rb, &dr) == CLS_OK && rb);
            cls_fasta_text *ft = nullptr;
            cls_fasta_host_records hr{};
            EXPECT(cls_fasta_read(reinterpret_cast<const uint8_t *>(text.data()), text.size(), &ft, &hr) == CLS_OK && hr.n_records == dr.n_records);
            if (rb && ft) {
                EXPECT(cls_place_resident(ix, rb, &params, nullptr) == CLS_OK);
                Results r(dr.n_records);
                cls_result rv = r.view();
                EXPECT(cls_resident_fetch(ix, rb, nullptr, &rv) == CLS_OK);
                Batch b;
                b.bases.assign(hr.bases, hr.bases + hr.offsets[hr.n_records]);
                b.offsets.assign(hr.offsets, hr.offsets + hr.n_records + 1);
                compare(b, r, orc, params, "fasta ingest");
            }
            if (rb) cls_resident_destroy(rb);
            if (ft) cls_fasta_text_destroy(ft);
        }
        cls_index_destroy(ix);
    }
    if (!threads_only) {
        // ---- 5. refusals ------------------------------------------------------------------------------------------------------
        const int devs[9] = {0, 1, 2, 0, 1, 2, 0, 1, 2};
        cls_index *ix = nullptr;
        EXPECT(cls_index_create_sharded(&model, 0, devs, &ix) == CLS_ERR_INVALID_ARGUMENT && !ix);
        EXPECT(cls_index_create_sharded(&model, 9, devs, &ix) == CLS_ERR_INVALID_ARGUMENT && !ix);
        setenv("FAKE_CUDA_NO_PEER", "1", 1);
        EXPECT(cls_index_create_sharded(&model, 2, devs, &ix) == CLS_ERR_UNSUPPORTED && !ix);
        const int same[2] = {1, 1};
        EXPECT(cls_index_create_sharded(&model, 2, same, &ix) == CLS_OK);   // one device: no peer access needed
        unsetenv("FAKE_CUDA_NO_PEER");
        Batch b = make_reads(300, 40, 161, 0);
        Batch longer = b;
        longer.add(std::string(162, 'A'));
        Results r(longer.n());
        cls_result rv = r.view();
        cls_batch lv = longer.view();
        EXPECT(cls_place_batch(ix, &lv, &params, &rv) == CLS_ERR_UNSUPPORTED && strstr(cls_last_error(), "161"));
        place(ix, b, params, "after the refused read");
        const cls_batch bv = b.view();
        cls_resident_batch *rb = nullptr;
        EXPECT(cls_batch_upload(ix, &bv, &rb) == CLS_OK);
        uint64_t nw = 0, counts[8];
        uint64_t rows = 0;
        std::vector<uint64_t> dummy(64);
        EXPECT(cls_routed_windows(ix, rb, &nw) == CLS_ERR_INVALID_ARGUMENT);
        EXPECT(cls_route_hashes(ix, rb, 2, 1024, dummy.data(), dummy.data(), counts, nullptr) == CLS_ERR_INVALID_ARGUMENT);
        void *segs[2] = {dummy.data(), dummy.data()};
        EXPECT(cls_route_hashes_p2p(ix, rb, 2, 1024, segs, dummy.data(), counts, nullptr) == CLS_ERR_INVALID_ARGUMENT);
        EXPECT(cls_shard_probe(ix, dummy.data(), 1, dummy.data(), nullptr) == CLS_ERR_INVALID_ARGUMENT);
        EXPECT(cls_place_routed(ix, rb, dummy.data(), dummy.data(), 2, 1024, &params, nullptr) == CLS_ERR_INVALID_ARGUMENT);
        EXPECT(cls_debug_node_counts(ix, b.bases.data(), 100, &params, nullptr, 0, &rows, nullptr) == CLS_ERR_INVALID_ARGUMENT);
        cls_resident_destroy(rb);
        cls_index_destroy(ix);

        // ---- 6. an allocation that fails at every position of create and of a placement: reported, nothing leaked ----------
        int failed = 0;
        for (long n = 1; n < 400; ++n) {
            const long before = fakecuda::live_allocs();
            fakecuda::fail_alloc_in() = n;
            cls_index *x = nullptr;
            const int rc = cls_index_create_sharded(&model, 3, devs, &x);
            const bool hit = fakecuda::fail_alloc_in().exchange(0) == 0;
            if (x) cls_index_destroy(x);
            EXPECT(hit == (rc != CLS_OK) && (rc == CLS_OK) == (x != nullptr) && fakecuda::live_allocs() == before);
            failed += hit;
            if (!hit) break;
        }
        const Batch small = make_reads(240, 30, 161, 0);
        for (int mode = 1; mode <= 2; ++mode) {
            cls_set_pack_mode(mode);
            for (long n = 1; n < 400; ++n) {
                const long before = fakecuda::live_allocs();
                cls_index *x = nullptr;
                EXPECT(cls_index_create_sharded(&model, 3, devs, &x) == CLS_OK);
                if (!x) break;
                Results res(small.n());
                cls_result sv = res.view();
                const cls_batch smv = small.view();
                fakecuda::fail_alloc_in() = n;
                const int rc = cls_place_batch(x, &smv, &params, &sv);
                cls_resident_batch *rb2 = nullptr;
                const int rc2 = rc == CLS_OK ? cls_batch_upload(x, &smv, &rb2) : CLS_OK;
                const int rc3 = rb2 ? cls_place_resident(x, rb2, &params, nullptr) : CLS_OK;
                const bool hit = fakecuda::fail_alloc_in().exchange(0) == 0;
                EXPECT(hit == (rc != CLS_OK || rc2 != CLS_OK || rc3 != CLS_OK));
                if (rb2) cls_resident_destroy(rb2);
                failed += hit;
                place(x, small, params, "after a failed allocation");   // memory is back: the handle works
                cls_index_destroy(x);
                EXPECT(fakecuda::live_allocs() == before);
                if (!hit) break;
            }
        }
        EXPECT(failed >= 40);
        // ---- 7. a CUDA call that reports an error, at every position of a placement: reported, the handle works after -----
        failed = 0;
        for (int mode = 1; mode <= 2; ++mode) {
            cls_set_pack_mode(mode);
            cls_index *x = nullptr;
            EXPECT(cls_index_create_sharded(&model, 3, devs, &x) == CLS_OK);
            for (long n = 1; n < 400 && x; ++n) {
                Results res(small.n());
                cls_result sv = res.view();
                const cls_batch smv = small.view();
                fakecuda::fail_call_in() = n;
                const int rc = cls_place_batch(x, &smv, &params, &sv);
                const bool hit = fakecuda::fail_call_in().exchange(0) == 0;
                EXPECT(hit == (rc != CLS_OK));
                failed += hit;
                place(x, small, params, "after a failed call");
                if (!hit) break;
            }
            cls_index_destroy(x);
        }
        cls_set_pack_mode(0);
        EXPECT(failed >= 40);
    }
    cls_index_destroy(flat);
    fakek::oracle_model = nullptr;
    orc_model_destroy(orc);
    cls_built_model_destroy(bm);
    EXPECT(fakek::async_errors == 0);
    EXPECT(fakecuda::live_allocs() == 0);
    printf("bad=%ld reads=%ld\n", g_bad.load(), g_reads.load());
    return g_bad == 0 && g_reads > (threads_only ? 10000 : 40000) ? 0 : 1;
}
