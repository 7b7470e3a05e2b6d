// TEST INFRASTRUCTURE.  cls_place_batch and its neighbours (classeq2_b200/csrc/place_batch.cpp) end to end WITHOUT a GPU: the
// library's host side is compiled against the fake CUDA runtime (tests/native/fakecuda/) and the placement launch hands
// the reads it was given - unpacked from the 2-bit words at their descriptors - to the C++ oracle
// (tests/native/fake_kernels.cpp).  The results must equal the oracle's on the caller's ASCII batch, for every way the
// host side can take: the just-in-time plan of short reads and its fallback, the general plan over many length classes,
// host / device / mixed packing from pageable and from pinned memory, many chunks, queries decided on the host (too
// short, invalid base), resident batches, the host side of the device FASTA ingest against the host reader, one handle over several devices, concurrent callers on one handle, a failing
// launch.  Built with AddressSanitizer + UBSan and with ThreadSanitizer by tests/test_capi_fake.py.
#include <atomic>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cmath>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include <cuda_runtime.h>
#include <unistd.h>

#include "../../include/classeq_b200.h"

namespace fakek {
extern const void *oracle_model;
extern std::atomic<uint64_t> place_launches, pack_launches, reads_placed, async_errors;
extern std::atomic<uint32_t> fail_above_len;
extern std::atomic<bool> null_placement;
}  // namespace fakek
extern "C" {
void *orc_model_create(const void *view);
void orc_model_destroy(void *);
void orc_place_batch(const void *model, const uint8_t *bases, const uint64_t *offsets, uint64_t n, int32_t max_iterations,
                     double min_match_coverage, uint32_t remove_intersection, int n_threads, uint8_t *status, uint64_t *node_id, int32_t *one,
                     int32_t *rest, uint32_t *n_query_kmers, uint32_t *n_matched, uint32_t *n_root_matched, uint32_t *iterations);
}

static uint64_t rng_state = 0x853C49E6748FEA9Bull;
static uint64_t rnd() { rng_state ^= rng_state << 13; rng_state ^= rng_state >> 7; rng_state ^= rng_state << 17; return rng_state; }

struct Results {
    std::vector<uint8_t> status; std::vector<uint64_t> node; std::vector<int32_t> one, rest; std::vector<uint32_t> nq, nm, nr, it;
    explicit Results(uint64_t n) : status(n, 0xEE), node(n, ~0ull), one(n, -7), rest(n, -7), nq(n, 77), nm(n, 77), nr(n, 77), it(n, 77) {}
    cls_result view() { return cls_result{status.data(), node.data(), one.data(), rest.data(), nq.data(), nm.data(), nr.data(), it.data()}; }
};

struct Batch {
    std::vector<uint8_t> bases;
    std::vector<uint64_t> offsets{0};
    uint64_t n() const { return offsets.size() - 1; }
    cls_batch view(const uint8_t *b = nullptr) const { return cls_batch{n(), b ? b : bases.data(), offsets.data()}; }
};

static long g_bad = 0, g_reads = 0;
#define EXPECT(c) do { if (!(c)) { ++g_bad; if (g_bad < 20) fprintf(stderr, "line %d: %s\n", __LINE__, #c); } } while (0)

static void compare(const Batch &b, Results &got, const void *orc, const cls_params &p, const char *what) {
    const uint64_t n = b.n();
    Results want(n);
    if (n) orc_place_batch(orc, b.bases.data(), b.offsets.data(), n, p.max_iterations, p.min_match_coverage, p.remove_intersection, 4,
                           want.status.data(), want.node.data(), want.one.data(), want.rest.data(), want.nq.data(), want.nm.data(),
                           want.nr.data(), want.it.data());
    long bad = 0;
    for (uint64_t i = 0; i < n; ++i) {
        bool invalid = false;
        for (uint64_t j = b.offsets[i]; j < b.offsets[i + 1]; ++j) { const uint8_t c = b.bases[j] & 0xDF; invalid |= !(c == 'A' || c == 'C' || c == 'G' || c == 'T'); }
        const uint64_t len = b.offsets[i + 1] - b.offsets[i];
        if (invalid && len >= 35) {   // decided on the host: the reference panics there (kmers_map.rs:440)
            bad += !(got.status[i] == CLS_STATUS_ERR_INVALID_BASE && got.node[i] == 0 && got.one[i] == 0 && got.rest[i] == 0 && got.nm[i] == 0 &&
                     got.nr[i] == 0 && got.it[i] == 0 && got.nq[i] == 2 * (len - 34));
            continue;
        }
        bad += !(got.status[i] == want.status[i] && got.node[i] == want.node[i] && got.one[i] == want.one[i] && got.rest[i] == want.rest[i] &&
                 got.nq[i] == want.nq[i] && got.nm[i] == want.nm[i] && got.nr[i] == want.nr[i] && got.it[i] == want.it[i]);
    }
    if (bad) fprintf(stderr, "%s: %ld of %llu queries differ\n", what, bad, (unsigned long long)n);
    g_bad += bad;
    g_reads += (long)n;
}

int main() {
    const int scale = 1;
    setenv("CLS_CHUNK_MBASES", "1", 1);           // 1 Mi bases per chunk: a few thousand reads are already several chunks
    setenv("CLS_HOST_THREADS", "4", 0);   // (not overwritten: a run with one thread takes the pool out)
    setenv("CLS_SEQ_BATCH", "3000", 1);           // cls_place_sequences: several batches, so that the writer overlaps a placement
    // ---- a model: random binary tree over 24 tips, sequences evolved along it, k = 35, m = 4 -----------------------------
    const uint32_t n_tips = 24;
    std::vector<uint64_t> node_id, child_off{0}, child_idx, tip_node;
    std::vector<uint8_t> kind;
    std::vector<std::string> seq_of_node;
    struct Todo { uint64_t node; uint32_t tips; };
    {
        std::vector<std::vector<uint64_t>> kids;
        std::vector<uint32_t> tips_below;
        auto add = [&](uint8_t k, const std::string &s, uint32_t t) { node_id.push_back(node_id.size() * 5 + 2); kind.push_back(k); seq_of_node.push_back(s); kids.emplace_back(); tips_below.push_back(t); return node_id.size() - 1; };
        std::string root_seq;
        for (int i = 0; i < 700; ++i) root_seq += "ACGT"[rnd() & 3];
        add(CLS_KIND_ROOT, root_seq, n_tips);
        for (uint64_t i = 0; i < node_id.size(); ++i) {                   // breadth first: children get larger indices
            if (tips_below[i] < 2) continue;
            const uint32_t left = 1 + (uint32_t)(rnd() % (tips_below[i] - 1));
            for (uint32_t part : {left, tips_below[i] - left}) {
                std::string s = seq_of_node[i];
                for (auto &c : s) if (rnd() % 40 == 0) c = "ACGT"[rnd() & 3];
                const uint64_t c = add(part == 1 ? CLS_KIND_LEAF : CLS_KIND_NODE, s, part);
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
    for (uint64_t t : tip_node) { refs.bases.insert(refs.bases.end(), seq_of_node[t].begin(), seq_of_node[t].end()); refs.offsets.push_back(refs.bases.size()); }
    cls_model_view tree{};
    tree.k_size = 35; tree.m_size = 4;
    tree.n_nodes = node_id.size(); tree.node_id = node_id.data(); tree.node_kind = kind.data(); tree.child_off = child_off.data(); tree.child_idx = child_idx.data();
    static const bool trace = getenv("CAPI_FAKE_TRACE") != nullptr;
#define STEP(what) do { if (trace) fprintf(stderr, "[capi_fake] %s\n", what); } while (0)
    STEP("model build");
    cls_built_model *bm = nullptr;
    if (cls_model_build(&tree, tip_node.size(), tip_node.data(), refs.bases.data(), refs.offsets.data(), &bm) != CLS_OK) { printf("model build failed: %s\n", cls_last_error()); return 1; }
    cls_model_view model{};
    cls_built_model_view(bm, &tree, &model);
    void *orc = orc_model_create(&model);
    fakek::oracle_model = orc;

    auto make_reads = [&](uint64_t n, uint32_t lo, uint32_t hi, int junk_every) {
        Batch b;
        for (uint64_t i = 0; i < n; ++i) {
            const std::string &s = seq_of_node[tip_node[rnd() % tip_node.size()]];
            uint32_t len = lo + (uint32_t)(rnd() % (hi - lo + 1));
            if (len > s.size()) len = (uint32_t)s.size();
            const uint32_t at = (uint32_t)(rnd() % (s.size() - len + 1));
            std::string r = rnd() % 20 == 0 ? std::string() : s.substr(at, len);
            if (r.empty()) for (uint32_t j = 0; j < len; ++j) r += "ACGT"[rnd() & 3];      // unrelated read
            for (auto &c : r) if (rnd() % 100 == 0) c = "ACGT"[rnd() & 3];
            if (rnd() % 2) for (auto &c : r) if (rnd() % 7 == 0) c = (char)(c | 0x20);        // lower case is valid input
            if (junk_every && i % junk_every == 3 && !r.empty()) r[rnd() % r.size()] = "NnX-*"[rnd() % 5];
            b.bases.insert(b.bases.end(), r.begin(), r.end());
            b.offsets.push_back(b.bases.size());
        }
        if (b.bases.empty()) b.bases.push_back('A');
        return b;
    };
    cls_params params;
    cls_params_default(&params);
    cls_index *ix = nullptr;
    STEP("index create");
    if (cls_index_create(&model, 0, &ix) != CLS_OK) { printf("index: %s\n", cls_last_error()); return 1; }

    // ---- 1. short reads (the just-in-time plan), every packing mode, pageable and pinned bases ---------------------------
    // (a chunk holds at least 4 096 reads: 9 000 reads are several chunks, 1 500 one)
    for (int mode = 1; mode <= 3; ++mode)
        for (int pin = 0; pin < 2; ++pin) {
            const Batch shorts = make_reads((mode == 2 && pin == 0) || (mode == 3 && pin == 1) ? 9000 : 1500, 36, 90, 0);   // (host packing over several chunks: scenario 2)
            void *pinned = nullptr;
            cudaHostAlloc(&pinned, shorts.bases.size(), cudaHostAllocDefault);
            memcpy(pinned, shorts.bases.data(), shorts.bases.size());
            cls_set_pack_mode(mode);
            STEP("1. short reads");
            Results r(shorts.n());
            cls_result rv = r.view();
            const cls_batch bv = shorts.view(pin ? static_cast<const uint8_t *>(pinned) : nullptr);
            EXPECT(cls_place_batch(ix, &bv, &params, &rv) == CLS_OK);
            compare(shorts, r, orc, params, "short reads");
            cls_timing tm{};
            EXPECT(cls_get_timing(ix, &tm) == CLS_OK && tm.kernel_launches >= 2 && tm.d2h_bytes >= 32 * shorts.n());
            EXPECT(tm.pack_on_device == (mode == 1 ? 0u : mode == 3 ? 3u : pin ? 2u : 1u));
            cudaFreeHost(pinned);
        }
    EXPECT(fakek::pack_launches > 0);
    // ---- 2. late in a batch of short reads: one read that is too short / too long (the just-in-time plan falls back to the
    //      general one), or reads with an invalid base (it does not: the packer that meets them flags them) ------
    for (int kind_of = 0; kind_of < 3; ++kind_of)
        for (int mode = 1 + kind_of % 2; mode <= 2; mode += 2) {
            cls_set_pack_mode(mode);
            Batch b = make_reads(4500, 40, 80, 0);   // (the first chunk holds 4 096 reads: the odd ones arrive while it is in flight)
            Batch odd = kind_of == 0 ? make_reads(1, 10, 20, 0) : kind_of == 1 ? make_reads(1, 300, 300, 0) : make_reads(8, 60, 60, 4);
            b.bases.insert(b.bases.end(), odd.bases.begin(), odd.bases.begin() + (long)odd.offsets.back());
            for (uint64_t i = 1; i < odd.offsets.size(); ++i) b.offsets.push_back(b.offsets[4500] + odd.offsets[i]);
            const Batch tail = make_reads(500, 40, 80, 0);
            const uint64_t base = b.offsets.back();
            b.bases.insert(b.bases.end(), tail.bases.begin(), tail.bases.end());
            for (uint64_t i = 1; i < tail.offsets.size(); ++i) b.offsets.push_back(base + tail.offsets[i]);
            Results r(b.n());
            cls_result rv = r.view();
            const cls_batch bv = b.view();
            EXPECT(cls_place_batch(ix, &bv, &params, &rv) == CLS_OK);
            compare(b, r, orc, params, "fallback");
        }
    // ---- 3. the general plan: lengths from below k to the whole reference, invalid bases here and there, both knob sets -----
    for (int mode = 1; mode <= 3; ++mode) {
        cls_set_pack_mode(mode);
        const Batch mixed = make_reads(2500 * scale, 1, 320, 11);
        cls_params p2 = params;
        p2.remove_intersection = mode == 2; p2.min_match_coverage = mode == 3 ? 0.2 : 0.7; p2.max_iterations = mode == 1 ? 2 : 1000;
        Results r(mixed.n());
        cls_result rv = r.view();
        const cls_batch bv = mixed.view();
        EXPECT(cls_place_batch(ix, &bv, &p2, &rv) == CLS_OK);
        compare(mixed, r, orc, p2, "mixed lengths");
        // the same batch resident: upload once, place twice, fetch
        cls_resident_batch *rb = nullptr;
        EXPECT(cls_batch_upload(ix, &bv, &rb) == CLS_OK);
        if (rb) {
            cudaStream_t user = nullptr;                                  // the caller's stream (bench.py hands a torch stream over)
            cudaStreamCreateWithFlags(&user, cudaStreamNonBlocking);
            EXPECT(cls_place_resident(ix, rb, &p2, user) == CLS_OK && cls_place_resident(ix, rb, &p2, user) == CLS_OK);
            Results r2(mixed.n());
            cls_result rv2 = r2.view();
            EXPECT(cls_resident_fetch(ix, rb, user, &rv2) == CLS_OK);
            compare(mixed, r2, orc, p2, "resident");
            cudaStreamDestroy(user);
            EXPECT(cls_resident_bytes(rb) > 0);
            cls_resident_destroy(rb);
        }
    }
    cls_set_pack_mode(0);
    // ---- 4. edges: no query, one query, only host-decided queries, result arrays that are partly NULL, bad arguments --------
    {
        Batch none;
        none.bases.push_back('A');
        Results r(0);
        cls_result rv = r.view();
        cls_batch bv = none.view();
        EXPECT(cls_place_batch(ix, &bv, &params, &rv) == CLS_OK);
        const Batch one = make_reads(1, 150, 150, 0);
        Results r1(1);
        cls_result rv1 = r1.view();
        bv = one.view();
        EXPECT(cls_place_batch(ix, &bv, &params, &rv1) == CLS_OK);
        compare(one, r1, orc, params, "one read");
        const Batch tiny = make_reads(300, 0, 34, 0);
        Results r2(tiny.n());
        cls_result rv2 = r2.view();
        bv = tiny.view();
        EXPECT(cls_place_batch(ix, &bv, &params, &rv2) == CLS_OK);
        compare(tiny, r2, orc, params, "too short");
        const Batch some = make_reads(1000, 40, 90, 0);
        Results r3(some.n());
        cls_result rv3 = r3.view();
        rv3.one = nullptr; rv3.n_matched = nullptr; rv3.iterations = nullptr;
        bv = some.view();
        EXPECT(cls_place_batch(ix, &bv, &params, &rv3) == CLS_OK);
        Results full(some.n());
        cls_result fv = full.view();
        EXPECT(cls_place_batch(ix, &bv, &params, &fv) == CLS_OK);
        EXPECT(r3.status == full.status && r3.node == full.node && r3.rest == full.rest && r3.one[5] == -7 && r3.it[5] == 77);
        std::vector<uint64_t> broken = some.offsets;
        std::swap(broken[100], broken[101]);
        cls_batch bb{some.n(), some.bases.data(), broken.data()};
        EXPECT(cls_place_batch(ix, &bb, &params, &fv) == CLS_ERR_INVALID_ARGUMENT);
        EXPECT(cls_place_batch(ix, nullptr, &params, &fv) == CLS_ERR_INVALID_ARGUMENT);
        bv = some.view();
        EXPECT(cls_place_batch(ix, &bv, &params, &fv) == CLS_OK);                 // the handle is as good as before
        compare(some, full, orc, params, "after the refused calls");
    }
    // ---- 5. a launch that fails: the call reports it, the workspace is given back, the next call works ---------------------
    {
        const Batch mixed = make_reads(1500, 40, 700, 0);
        Results r(mixed.n());
        cls_result rv = r.view();
        const cls_batch bv = mixed.view();
        fakek::fail_above_len = 500;
        EXPECT(cls_place_batch(ix, &bv, &params, &rv) == CLS_ERR_UNSUPPORTED);
        fakek::fail_above_len = 0;
        EXPECT(cls_place_batch(ix, &bv, &params, &rv) == CLS_OK);
        compare(mixed, r, orc, params, "after a failed launch");
    }
    // ---- 5b. FASTA ingest "on the device": cls_fasta_upload's host side (record rules over the per-header-line facts,
    //      header ends, planning) against the host reader cls_fasta_read - same records, same placements -------------------------
    for (int t = 0; t < 40; ++t) {
        std::string text;
        const int n_rec = (int)(rnd() % 60);
        const char *eol = t % 3 == 1 ? "\r\n" : "\n";
        for (int i = 0; i < n_rec; ++i) {
            if (!(t % 7 == 3 && i == 0)) {                                      // t % 7 == 3: sequence before the first header
                text += rnd() % 9 == 0 ? ">>" : ">";
                if (rnd() % 11) text += "read_" + std::to_string(i) + (rnd() % 3 ? "" : " some>text");   // else: an empty header
                text += eol;
            }
            const Batch one = make_reads(1, 20, 260, 0);
            std::string body(one.bases.begin(), one.bases.begin() + (long)one.offsets[1]);
            if (rnd() % 12 == 0) body.clear();
            for (size_t a = 0; a < body.size();) {                               // wrapped lines with junk the filter deletes
                const size_t w = 1 + rnd() % 90;
                text += body.substr(a, w);
                if (rnd() % 5 == 0) text += "NN--  xyz";
                text += eol;
                if (rnd() % 13 == 0) text += eol;
                a += w;
            }
        }
        if (t % 5 == 0 && !text.empty()) text.pop_back();                        // no final newline
        cls_fasta_text *ft = nullptr;
        cls_fasta_host_records hr{};
        EXPECT(cls_fasta_read(reinterpret_cast<const uint8_t *>(text.data()), text.size(), &ft, &hr) == CLS_OK);
        cls_resident_batch *rb = nullptr;
        cls_fasta_records dr{};
        EXPECT(cls_fasta_upload(ix, reinterpret_cast<const uint8_t *>(text.data()), text.size(), &rb, &dr) == CLS_OK);
        if (!ft || !rb) { ++g_bad; continue; }
        EXPECT(dr.n_records == hr.n_records);
        Batch b;
        b.bases.assign(hr.bases, hr.bases + hr.offsets[hr.n_records]);
        if (b.bases.empty()) b.bases.push_back('A');
        b.offsets.assign(hr.offsets, hr.offsets + hr.n_records + 1);
        for (uint64_t i = 0; i < hr.n_records && i < dr.n_records; ++i)
            EXPECT(dr.header_begin[i] == hr.header_begin[i] && dr.header_end[i] == hr.header_end[i] && dr.length[i] == hr.offsets[i + 1] - hr.offsets[i]);
        Results r(dr.n_records);
        cls_result rv = r.view();
        EXPECT(cls_place_resident(ix, rb, &params, nullptr) == CLS_OK && cls_resident_fetch(ix, rb, nullptr, &rv) == CLS_OK);
        if (dr.n_records == hr.n_records) compare(b, r, orc, params, "fasta upload");
        cls_resident_destroy(rb);
        cls_fasta_text_destroy(ft);
    }
    {   // a non-ASCII byte: refused, the host reader takes such files
        const std::string text = ">a\nACGT\xC3\xA9" "ACGT\n";
        cls_resident_batch *rb = nullptr;
        cls_fasta_records dr{};
        EXPECT(cls_fasta_upload(ix, reinterpret_cast<const uint8_t *>(text.data()), text.size(), &rb, &dr) == CLS_ERR_UNSUPPORTED && !rb);
    }
    // ---- 5c. the whole use-case in one call: cls_place_sequences = reader + the REAL cls_place_batch per batch of 3 000 queries
    //      + the writer, which renders and appends batch i on a second thread while batch i + 1 is placed ------------------------------
    if (fakecuda::async()) {                  // (a scenario about threads: the runs with asynchronous streams take it)
        STEP("5c. cls_place_sequences");
        const uint64_t nn = node_id.size();
        std::vector<int64_t> parent_id(nn, -1);
        for (uint64_t i = 0; i < nn; ++i) for (uint64_t j = child_off[i]; j < child_off[i + 1]; ++j) parent_id[child_idx[j]] = (int64_t)node_id[i];
        std::vector<uint8_t> children_some(nn), has_name(nn);
        std::vector<double> support(nn), length(nn);
        std::vector<uint64_t> name_off{0};
        std::string names;
        for (uint64_t i = 0; i < nn; ++i) {
            children_some[i] = kind[i] != CLS_KIND_LEAF;
            has_name[i] = kind[i] == CLS_KIND_LEAF;
            if (has_name[i]) names += "tip_" + std::to_string(i);
            name_off.push_back(names.size());
            support[i] = kind[i] == CLS_KIND_NODE ? 70.0 + (double)(i % 30) : NAN;
            length[i] = 0.001 * (double)(i + 1);
        }
        const uint64_t no_ann[2] = {0, 0};
        cls_record_tree rt{};
        rt.n_nodes = nn; rt.node_id = node_id.data(); rt.parent_id = parent_id.data(); rt.node_kind = kind.data(); rt.children_some = children_some.data();
        rt.support = support.data(); rt.length = length.data(); rt.has_name = has_name.data(); rt.name_off = name_off.data(); rt.names = names.data();
        rt.child_off = child_off.data(); rt.child_idx = child_idx.data();
        rt.ann_clade = no_ann; rt.ann_yaml_off = no_ann; rt.ann_yaml = ""; rt.ann_json_off = no_ann; rt.ann_json = "";
        const Batch reads = make_reads(10000, 20, 120, 0);                       // some below k: lines of the error file
        std::string fasta, headers;
        std::vector<uint64_t> header_off{0};
        for (uint64_t i = 0; i < reads.n(); ++i) {
            const std::string h = "q" + std::to_string(i) + (i % 3 ? "" : " with text");
            if (reads.offsets[i + 1] == reads.offsets[i]) continue;             // (make_reads never makes one; the reader would drop a trailing one)
            fasta += ">" + h + "\n";
            fasta.append(reads.bases.begin() + (long)reads.offsets[i], reads.bases.begin() + (long)reads.offsets[i + 1]);
            fasta += "\n";
            headers += h;
            header_off.push_back(headers.size());
        }
        char dir[] = "/tmp/capi_fake_XXXXXX";
        if (!mkdtemp(dir)) { printf("mkdtemp failed\n"); return 1; }
        const std::string in = std::string(dir) + "/in.fasta", out = std::string(dir) + "/res.x";
        FILE *f = fopen(in.c_str(), "wb");
        fwrite(fasta.data(), 1, fasta.size(), f);
        fclose(f);
        for (uint32_t fmt = 0; fmt < 2; ++fmt) {
            uint64_t placed = 0;
            EXPECT(cls_place_sequences(ix, &rt, in.c_str(), out.c_str(), &params, fmt, 1, &placed) == CLS_OK && placed == reads.n());
            // expected: one cls_place_batch over everything (upper-cased, as the reader hands it over) + one render
            Batch up = reads;
            for (auto &c : up.bases) c &= 0xDF;
            Results r(up.n());
            cls_result rv = r.view();
            const cls_batch bv = up.view();
            EXPECT(cls_place_batch(ix, &bv, &params, &rv) == CLS_OK);
            compare(up, r, orc, params, "place_sequences: the batch");
            char *ot = nullptr, *et = nullptr;
            uint64_t ol = 0, el = 0;
            EXPECT(cls_records_render(&rt, up.n(), header_off.data(), headers.data(), &rv, fmt, &ot, &ol, &et, &el) == CLS_OK);
            auto slurp = [](const std::string &p) { std::string t; FILE *g = fopen(p.c_str(), "rb"); if (!g) return t; char buf[65536]; size_t k; while ((k = fread(buf, 1, sizeof buf, g)) > 0) t.append(buf, k); fclose(g); return t; };
            const std::string got_o = slurp(std::string(dir) + (fmt ? "/res.jsonl" : "/res.yaml")), got_e = slurp(std::string(dir) + "/res.error");
            EXPECT(ot && got_o == std::string(ot, ol) && ol > 100000);
            EXPECT(et && got_e.size() >= el && got_e.compare(got_e.size() - el, el, et, el) == 0 && el > 0);   // the error file is appended to
            cls_text_free(ot); cls_text_free(et);
        }
        for (const char *n : {"/in.fasta", "/res.yaml", "/res.jsonl", "/res.error"}) remove((std::string(dir) + n).c_str());
        rmdir(dir);
    }
    STEP("6. concurrent callers");
    // ---- 6. concurrent callers on one handle (per-call workspaces) -------------------------------------------------------------
    {
        std::vector<Batch> bs;
        for (int t = 0; t < 4; ++t) bs.push_back(make_reads(1200, t % 2 ? 30 : 40, t % 2 ? 250 : 90, t == 3 ? 9 : 0));
        std::vector<Results> rs;
        for (auto &b : bs) rs.emplace_back(b.n());
        std::vector<std::thread> th;
        std::atomic<int> failed{0};
        for (int t = 0; t < 4; ++t)
            th.emplace_back([&, t] {
                for (int rep = 0; rep < 2; ++rep) {
                    cls_result rv = rs[t].view();
                    const cls_batch bv = bs[t].view();
                    if (cls_place_batch(ix, &bv, &params, &rv) != CLS_OK) ++failed;
                }
            });
        for (auto &t : th) t.join();
        EXPECT(failed == 0);
        for (int t = 0; t < 4; ++t) compare(bs[t], rs[t], orc, params, "concurrent callers");
    }
    cls_index_destroy(ix);
    STEP("7. three devices");
    // ---- 7. one handle over three devices: the batch is cut by bases, the parts run side by side ----------------------------------
    {
        cls_index *multi = nullptr;
        EXPECT(cls_index_create_multi(&model, 0b1011, &multi) == CLS_OK);
        cls_index_info info{};
        EXPECT(multi && cls_index_get_info(multi, &info) == CLS_OK && info.n_devices == 3);
        EXPECT(cls_index_create_multi(&model, 1ull << 9, &ix) != CLS_OK);             // no such device
        if (multi) {
            for (int round = 0; round < 3; ++round) {
                const Batch b = round == 0 ? make_reads(9000 * scale, 36, 90, 0) : round == 1 ? make_reads(2500, 1, 320, 13) : make_reads(2, 150, 150, 0);
                Results r(b.n());
                cls_result rv = r.view();
                const cls_batch bv = b.view();
                cls_set_pack_mode(round == 1 ? 2 : 0);
                EXPECT(cls_place_batch(multi, &bv, &params, &rv) == CLS_OK);
                compare(b, r, orc, params, "three devices");
            }
            cls_set_pack_mode(0);
            cls_index_destroy(multi);
        }
    }
    // ---- 8. an allocation that fails (device or pinned), at every position in turn: the call reports it, nothing is leaked,
    //      and the same handle places the batch once memory is back -----------------------------------------------------------------
    if (!fakecuda::async()) {
        STEP("8. failing allocations");
        const Batch b = make_reads(40, 30, 300, 7);
        const cls_batch bv = b.view();
        int failed_creates = 0, failed_calls = 0;
        for (long n = 1; n < 200; ++n) {                                    // cls_index_create
            const long before = fakecuda::live_allocs();
            fakecuda::fail_alloc_in() = n;
            cls_index *x = nullptr;
            const int rc = cls_index_create(&model, 1, &x);
            const bool hit = fakecuda::fail_alloc_in().exchange(0) == 0;     // the failure was consumed
            if (!hit) { EXPECT(rc == CLS_OK && x); cls_index_destroy(x); EXPECT(fakecuda::live_allocs() == before); break; }
            EXPECT(rc != CLS_OK && !x && cls_last_error()[0] != 0);
            EXPECT(fakecuda::live_allocs() == before);
            ++failed_creates;
        }
        for (long n = 1; n < 200; ++n) {                                    // one handle over three devices: the replicas made so far are released
            const long before = fakecuda::live_allocs();
            fakecuda::fail_alloc_in() = n;
            cls_index *x = nullptr;
            const int rc = cls_index_create_multi(&model, 0b111, &x);
            const bool hit = fakecuda::fail_alloc_in().exchange(0) == 0;
            if (x) cls_index_destroy(x);
            EXPECT(hit == (rc != CLS_OK) && (rc == CLS_OK) == (x != nullptr) && fakecuda::live_allocs() == before);
            failed_creates += hit;
            if (!hit) break;
        }
        {                                                                   // cls_fasta_upload: its temporaries and the batch it was building
            const std::string text = ">a\nACGTTGCAAGCTTGCATGCCTGCAGGTCGACTCTAGAGGATCCCCGGGTACCGAGCTCGAATTC\n>b\nACGTTGCAAGCTTGCATGCCTGCAGGTCGACTCTAGAGGATCCCC\n";
            cls_index *x = nullptr;
            EXPECT(cls_index_create(&model, 0, &x) == CLS_OK);
            for (long n = 1; n < 200 && x; ++n) {
                const long before = fakecuda::live_allocs();
                fakecuda::fail_alloc_in() = n;
                cls_resident_batch *rb = nullptr;
                cls_fasta_records dr{};
                const int rc = cls_fasta_upload(x, reinterpret_cast<const uint8_t *>(text.data()), text.size(), &rb, &dr);
                const bool hit = fakecuda::fail_alloc_in().exchange(0) == 0;
                EXPECT(hit == (rc != CLS_OK) && (rc == CLS_OK) == (rb != nullptr));
                if (rb) { EXPECT(dr.n_records == 2); cls_resident_destroy(rb); }
                EXPECT(fakecuda::live_allocs() == before);
                failed_calls += hit;
                if (!hit) break;
            }
            cls_index_destroy(x);
        }
        for (int mode = 1; mode <= 2; ++mode) {                             // cls_place_batch and the resident calls, host and device packing
            cls_set_pack_mode(mode);
            for (long n = 1; n < 200; ++n) {
                cls_index *x = nullptr;
                EXPECT(cls_index_create(&model, 2, &x) == CLS_OK);
                if (!x) break;
                Results r(b.n());
                cls_result rv = r.view();
                fakecuda::fail_alloc_in() = n;
                const int rc = cls_place_batch(x, &bv, &params, &rv);
                cls_resident_batch *rb = nullptr;
                const int rc2 = rc == CLS_OK ? cls_batch_upload(x, &bv, &rb) : CLS_OK;
                const int rc3 = rb ? cls_place_resident(x, rb, &params, nullptr) : CLS_OK;
                const int rc4 = rb && rc3 == CLS_OK ? cls_resident_fetch(x, rb, nullptr, &rv) : CLS_OK;
                const bool hit = fakecuda::fail_alloc_in().exchange(0) == 0;
                EXPECT(hit == (rc != CLS_OK || rc2 != CLS_OK || rc3 != CLS_OK || rc4 != CLS_OK));
                failed_calls += hit;
                if (rb) cls_resident_destroy(rb);
                Results again(b.n());
                cls_result av = again.view();
                EXPECT(cls_place_batch(x, &bv, &params, &av) == CLS_OK);    // memory is back: the handle works
                compare(b, again, orc, params, "after a failed allocation");
                cls_index_destroy(x);
                if (!hit) break;
            }
        }
        cls_set_pack_mode(0);
        EXPECT(failed_creates >= 30 && failed_calls >= 20);
    }
    // ---- 9. a CUDA call that reports an error, at every position of a call of several chunks in turn: the call reports it and
    //      leaves NOTHING in flight on its workspace - the very next call on the handle takes the same workspace and must give
    //      the same results (with asynchronous streams a copy or a launch that outlived the failed call would race with it).
    //      The launches write "no match" records here: what is compared is one call against another --------------------------------
    {
        STEP("9. failing CUDA calls");
        fakek::null_placement = true;
        const Batch b = make_reads(9000, 36, 90, 0);
        const cls_batch bv = b.view();
        int failed_calls = 0;
        for (int mode = 1; mode <= 2; ++mode) {
            cls_set_pack_mode(mode);
            cls_index *x = nullptr;
            EXPECT(cls_index_create(&model, 0, &x) == CLS_OK);
            if (!x) break;
            Results ref(b.n());
            cls_result refv = ref.view();
            EXPECT(cls_place_batch(x, &bv, &params, &refv) == CLS_OK);
            for (long n = 1; n < 400; ++n) {
                Results r(b.n());
                cls_result rv = r.view();
                fakecuda::fail_call_in() = n;
                const int rc = cls_place_batch(x, &bv, &params, &rv);
                const bool hit = fakecuda::fail_call_in().exchange(0) == 0;
                EXPECT(hit == (rc != CLS_OK));
                failed_calls += hit;
                Results again(b.n());
                cls_result av = again.view();
                EXPECT(cls_place_batch(x, &bv, &params, &av) == CLS_OK);
                EXPECT(again.status == ref.status && again.node == ref.node && again.nq == ref.nq && again.nm == ref.nm);
                if (!hit) break;
            }
            cls_index_destroy(x);
        }
        cls_set_pack_mode(0);
        fakek::null_placement = false;
        EXPECT(failed_calls >= 40);
    }
    fakek::oracle_model = nullptr;
    orc_model_destroy(orc);
    cls_built_model_destroy(bm);
    EXPECT(fakek::async_errors == 0);
    EXPECT(fakecuda::live_allocs() == 0);                                                // every device / pinned buffer was released
    printf("bad=%ld reads=%ld place_launches=%llu pack_launches=%llu\n", g_bad, g_reads, (unsigned long long)fakek::place_launches.load(),
           (unsigned long long)fakek::pack_launches.load());
    return g_bad == 0 && g_reads > 50000 ? 0 : 1;
}
