// TEST INFRASTRUCTURE.  The host side of cls_fastq_upload (classeq2_b200/csrc/fastq_ingest.cpp, capi.cu) WITHOUT a GPU: compiled against the
// fake CUDA runtime (tests/native/fakecuda/), with fastq_kernels.cu's launches restated as serial walks
// (fake_fastq_kernels.cpp) and the placement launch answered by the C++ oracle (fake_kernels.cpp).  On random and
// hand-made FASTQ texts the upload must give cls_fastq_read's records (header slices, lengths) and the placements
// cls_place_batch gives on the reader's bases; a malformed text must be refused with the reader's message and leave no
// batch and no buffer behind.  Built with AddressSanitizer + UBSan by tests/test_fastq_ingest.py.
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include <cuda_runtime.h>

#include "../../include/classeq_b200.h"

namespace fakek {
extern const void *oracle_model;
}
extern "C" {
void *orc_model_create(const void *view);
void orc_model_destroy(void *);
}

static uint64_t rng_state = 0x2545F4914F6CDD1Dull;
static uint64_t rnd() { rng_state ^= rng_state << 13; rng_state ^= rng_state >> 7; rng_state ^= rng_state << 17; return rng_state; }

static long g_bad = 0, g_records = 0;
#define EXPECT(c) do { if (!(c)) { ++g_bad; if (g_bad < 20) fprintf(stderr, "line %d: %s\n", __LINE__, #c); } } while (0)

struct Results {
    std::vector<uint8_t> status; std::vector<uint64_t> node; std::vector<int32_t> one, rest; std::vector<uint32_t> nq, nm, nr, it;
    explicit Results(uint64_t n) : status(n, 0xEE), node(n, ~0ull), one(n, -7), rest(n, -7), nq(n, 77), nm(n, 77), nr(n, 77), it(n, 77) {}
    cls_result view() { return cls_result{status.data(), node.data(), one.data(), rest.data(), nq.data(), nm.data(), nr.data(), it.data()}; }
    bool operator==(const Results &o) const {
        return status == o.status && node == o.node && one == o.one && rest == o.rest && nq == o.nq && nm == o.nm && nr == o.nr && it == o.it;
    }
};

// One text through both readers: the same records and placements, or the same refusal.
static void check(cls_index *ix, const std::string &text, const cls_params &params) {
    const uint8_t *t = reinterpret_cast<const uint8_t *>(text.data());
    cls_fasta_text *ft = nullptr;
    cls_fasta_host_records hr{};
    const int hrc = cls_fastq_read(t, text.size(), &ft, &hr);
    const std::string herr = hrc == CLS_OK ? "" : cls_last_error();
    cls_resident_batch *rb = nullptr;
    cls_fasta_records dr{};
    const int drc = cls_fastq_upload(ix, t, text.size(), &rb, &dr);
    EXPECT(drc == hrc);
    if (hrc != CLS_OK || drc != CLS_OK) {
        EXPECT(!rb && !ft && herr == cls_last_error());
        cls_resident_destroy(rb);
        cls_fasta_text_destroy(ft);
        return;
    }
    EXPECT(dr.n_records == hr.n_records);
    const uint64_t n = dr.n_records < hr.n_records ? dr.n_records : hr.n_records;
    for (uint64_t i = 0; i < n; ++i)
        EXPECT(dr.header_begin[i] == hr.header_begin[i] && dr.header_end[i] == hr.header_end[i] && dr.length[i] == hr.offsets[i + 1] - hr.offsets[i]);
    if (dr.n_records == hr.n_records) {
        Results got(n), want(n);
        cls_result gv = got.view(), wv = want.view();
        std::vector<uint8_t> bases(hr.bases, hr.bases + hr.offsets[n]);
        if (bases.empty()) bases.push_back('A');
        const cls_batch b{n, bases.data(), hr.offsets};
        EXPECT(cls_place_resident(ix, rb, &params, nullptr) == CLS_OK && cls_resident_fetch(ix, rb, nullptr, &gv) == CLS_OK);
        EXPECT(cls_place_batch(ix, &b, &params, &wv) == CLS_OK);
        EXPECT(got == want);
        g_records += (long)n;
    }
    cls_resident_destroy(rb);
    cls_fasta_text_destroy(ft);
}

int main() {
    setenv("CLS_HOST_THREADS", "4", 0);
    // ---- a model: 12 tips, each a mutated copy of one random root sequence, on a comb tree; k = 35, m = 4 -----------------
    const uint32_t n_tips = 12;
    std::string root_seq;
    for (int i = 0; i < 600; ++i) root_seq += "ACGT"[rnd() & 3];
    std::vector<uint64_t> node_id, child_off{0}, child_idx, tip_node;
    std::vector<uint8_t> kind;
    std::vector<std::string> tips;
    // node 0 = root, nodes 1..n_tips = leaves under it
    node_id.push_back(7); kind.push_back(CLS_KIND_ROOT);
    for (uint32_t t = 0; t < n_tips; ++t) {
        node_id.push_back(100 + t); kind.push_back(CLS_KIND_LEAF); child_idx.push_back(1 + t); tip_node.push_back(1 + t);
        std::string s = root_seq;
        for (auto &c : s) if (rnd() % 15 == 0) c = "ACGT"[rnd() & 3];
        tips.push_back(s);
    }
    child_off.push_back(n_tips);
    for (uint32_t t = 0; t < n_tips; ++t) child_off.push_back(n_tips);
    std::vector<uint8_t> ref_bases;
    std::vector<uint64_t> ref_off{0};
    for (const auto &s : tips) { ref_bases.insert(ref_bases.end(), s.begin(), s.end()); ref_off.push_back(ref_bases.size()); }
    cls_model_view tree{};
    tree.k_size = 35; tree.m_size = 4;
    tree.n_nodes = node_id.size(); tree.node_id = node_id.data(); tree.node_kind = kind.data(); tree.child_off = child_off.data(); tree.child_idx = child_idx.data();
    cls_built_model *bm = nullptr;
    if (cls_model_build(&tree, tip_node.size(), tip_node.data(), ref_bases.data(), ref_off.data(), &bm) != CLS_OK) { printf("model build failed: %s\n", cls_last_error()); return 1; }
    cls_model_view model{};
    cls_built_model_view(bm, &tree, &model);
    void *orc = orc_model_create(&model);
    fakek::oracle_model = orc;
    cls_index *ix = nullptr;
    if (cls_index_create(&model, 0, &ix) != CLS_OK) { printf("index: %s\n", cls_last_error()); return 1; }
    cls_params params;
    cls_params_default(&params);

    // ---- random texts: reads cut from the tips, junk the filter deletes, CRLF, quality lines starting with '@' / '+', empty
    //      and short sequences, titles with '>' / '@' / UTF-8, trailing blank lines, no final newline ----------------------
    for (int t = 0; t < 60; ++t) {
        std::string text;
        const int n_rec = (int)(rnd() % 80);
        const char *eol = t % 3 == 1 ? "\r\n" : "\n";
        for (int i = 0; i < n_rec; ++i) {
            const std::string &s = tips[rnd() % n_tips];
            const size_t len = rnd() % 12 == 0 ? rnd() % 40 : 30 + rnd() % 500;
            const size_t at = rnd() % (s.size() - (len < s.size() ? len : s.size()) + 1);
            std::string seq = s.substr(at, len);
            for (auto &c : seq) if (rnd() % 9 == 0) c = (char)(c | 0x20);
            if (rnd() % 4 == 0 && !seq.empty()) seq.insert(rnd() % seq.size(), rnd() % 2 ? "NN-." : "\xC3\xA9");
            std::string title = "r" + std::to_string(i);
            if (rnd() % 10 == 0) title += " x>y@z";
            if (rnd() % 15 == 0) title += " \xE2\x82\xAC";
            if (rnd() % 30 == 0) title.clear();
            std::string qual(seq.size(), 'I');
            if (!qual.empty() && rnd() % 8 == 0) qual[0] = rnd() % 2 ? '@' : '+';
            text += "@" + title + eol + seq + eol + (rnd() % 5 ? "+" : "+" + title) + eol + qual + eol;
        }
        if (t % 7 == 2) text += "\n\r\n\n";
        if (t % 5 == 0 && !text.empty()) text.pop_back();
        if (t % 11 == 4) {                                                        // a malformed record somewhere: the same refusal
            const size_t cut = text.empty() ? 0 : rnd() % text.size();
            const char *bad[] = {"\n@x\nAC\n+\nI\n", "\n\n@x\nAC\n+\nII\n", "\n@x\xFF\nAC\n+\nII\n", "\nx\nAC\n+\nII\n"};
            text.insert(cut, bad[rnd() % 4]);
        }
        check(ix, text, params);
    }
    for (const char *text : {"", "\n\n", "@a\nACGT\n+\nIIII", "@a\nACGT\n+\nIII\n", "@a\nACGT\n", "@\n\n+\n\n", "@a\r\nAC\r\n+\r\nI\r",
                             "@a\nACGT\n+\nIIII\n\n@b\nA\n+\nI\n", "@a\xC3\nACGT\n+\nIIII\n", "@a\nAC\n-\nII\n@b\xFF\nA\n+\nI\n"})
        check(ix, text, params);
    {   // an upload whose placement is never run, then a text of 4 GiB is refused before anything is read
        cls_resident_batch *rb = nullptr;
        cls_fasta_records dr{};
        const std::string text = "@a\nACGTACGTACGTACGTACGTACGTACGTACGTACGTACGT\n+\nIIIIIIIIIIIIIIIIIIIIIIIIIIIIIIIIIIIIIIII\n";
        EXPECT(cls_fastq_upload(ix, reinterpret_cast<const uint8_t *>(text.data()), text.size(), &rb, &dr) == CLS_OK && dr.n_records == 1);
        cls_resident_destroy(rb);
        rb = nullptr;
        EXPECT(cls_fastq_upload(ix, reinterpret_cast<const uint8_t *>(text.data()), 1ull << 32, &rb, &dr) == CLS_ERR_UNSUPPORTED && !rb);
        EXPECT(strncmp(cls_last_error(), "FASTQ text of 4 GiB or more", 27) == 0);
    }
    cls_index_destroy(ix);
    fakek::oracle_model = nullptr;
    orc_model_destroy(orc);
    cls_built_model_destroy(bm);
    EXPECT(fakecuda::live_allocs() == 0);   // every device / pinned buffer was released, on the refusals too
    printf("bad=%ld records=%ld\n", g_bad, g_records);
    return g_bad == 0 && g_records > 1000 ? 0 : 1;
}
