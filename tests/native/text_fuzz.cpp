// TEST INFRASTRUCTURE.  Memory-safety fuzz of the library's host text code (classeq2_b200/csrc/record_writer.cpp:
// cls_fasta_read, cls_filter_sequence, cls_records_render) under AddressSanitizer + UndefinedBehaviorSanitizer: random
// FASTA-like byte soup (every byte value, odd line ends, '>' everywhere) and random trees / names / statuses.  It checks
// invariants (offsets monotone, only A/C/G/T kept, headers inside the text), not output equality - that is what
// tests/test_fasta_reader.py and tests/test_record_writer.py do.  Built and run by tests/test_text_fuzz.py.
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <string>
#include <vector>

#include "../../include/classeq_b200.h"

namespace cls {
int set_last_error(int code, const std::string &) { return code; }   // capi.cpp's, stubbed
}
extern "C" int cls_place_batch(cls_index *, const cls_batch *, const cls_params *, cls_result *) { return CLS_ERR_CUDA; }  // no device here
extern "C" const char *cls_last_error(void) { return ""; }   // capi.cpp's (cls_place_sequences carries the writer thread's message over)

static uint64_t rng_state = 88172645463325252ull;
static uint64_t rnd() { rng_state ^= rng_state << 13; rng_state ^= rng_state >> 7; rng_state ^= rng_state << 17; return rng_state; }

static std::string soup(size_t n, int flavour) {
    static const char common[] = "ACGTacgtNn>\n\r\n \t-";
    std::string s;
    for (size_t i = 0; i < n; ++i) {
        const uint64_t r = rnd();
        if (flavour == 0 || (r & 7) == 0) s += (char)(rnd() & 0xFF);
        else s += common[(r >> 8) % (sizeof common - 1)];
    }
    return s;
}

int main(int argc, char **argv) {
    const int rounds = argc > 1 ? atoi(argv[1]) : 300;
    long bad = 0;
    for (int r = 0; r < rounds; ++r) {
        // ---- reader
        const std::string text = soup(rnd() % 3000, r % 3);
        cls_fasta_text *h = nullptr;
        cls_fasta_host_records rec;
        setenv("CLS_FASTA_CHUNK", std::to_string(1 + rnd() % 200).c_str(), 1);   // chunks of a few lines: the stitching pass sees every rule
        if (cls_fasta_read(reinterpret_cast<const uint8_t *>(text.data()), text.size(), &h, &rec) != CLS_OK) { ++bad; continue; }
        {   // ... and gives what one chunk gives
            setenv("CLS_FASTA_CHUNK", "1000000000", 1);
            cls_fasta_text *h1 = nullptr;
            cls_fasta_host_records r1;
            if (cls_fasta_read(reinterpret_cast<const uint8_t *>(text.data()), text.size(), &h1, &r1) != CLS_OK) { ++bad; continue; }
            if (r1.n_records != rec.n_records) ++bad;
            else {
                for (uint64_t i = 0; i < rec.n_records; ++i)
                    if (r1.header_begin[i] != rec.header_begin[i] || r1.header_end[i] != rec.header_end[i] || r1.offsets[i + 1] != rec.offsets[i + 1]) ++bad;
                for (uint64_t j = 0; j < rec.offsets[rec.n_records]; ++j)
                    if (r1.bases[j] != rec.bases[j]) ++bad;
            }
            cls_fasta_text_destroy(h1);
        }
        for (uint64_t i = 0; i < rec.n_records; ++i) {
            if (rec.offsets[i] > rec.offsets[i + 1] || rec.header_begin[i] >= rec.header_end[i] || rec.header_end[i] > text.size()) ++bad;
            if (text[rec.header_begin[i]] != '>') ++bad;
            for (uint64_t j = rec.offsets[i]; j < rec.offsets[i + 1]; ++j) {
                const uint8_t c = rec.bases[j];
                if (c != 'A' && c != 'C' && c != 'G' && c != 'T') ++bad;
            }
        }
        // ---- writer: a random tree whose names are pieces of the soup, results with every status
        const uint64_t n_nodes = 1 + rnd() % 40;
        std::vector<uint64_t> node_id(n_nodes), child_off(n_nodes + 1, 0), child_idx, name_off(n_nodes + 1, 0);
        std::vector<int64_t> parent_id(n_nodes);
        std::vector<uint8_t> kind(n_nodes), children_some(n_nodes), has_name(n_nodes);
        std::vector<double> support(n_nodes), length(n_nodes);
        std::string names;
        std::vector<std::vector<uint64_t>> kids(n_nodes);
        for (uint64_t i = 0; i < n_nodes; ++i) {
            node_id[i] = rnd() % 3 ? i : rnd() % 50;                     // duplicated ids happen
            const uint64_t p = i ? rnd() % i : 0;
            if (i) kids[p].push_back(i);
            parent_id[i] = i == 0 ? -1 : (rnd() % 5 ? (int64_t)node_id[p] : (int64_t)(rnd() % 60));   // parent FIELDS may lie
            kind[i] = i == 0 ? CLS_KIND_ROOT : (rnd() % 2 ? CLS_KIND_LEAF : CLS_KIND_NODE);
            has_name[i] = rnd() % 2;
            const std::string nm = has_name[i] ? soup(rnd() % 30, 1) : std::string();
            names += nm;
            name_off[i + 1] = names.size();
            const double vals[] = {0.0, -0.0, 1e-6, 72.0, 1e16, NAN, INFINITY, -1.5e-300, 5e-324, 123456.789};
            support[i] = vals[rnd() % 10];
            length[i] = vals[rnd() % 10];
        }
        for (uint64_t i = 0; i < n_nodes; ++i) {
            children_some[i] = !kids[i].empty() || rnd() % 2;
            for (uint64_t c : kids[i]) child_idx.push_back(c);
            child_off[i + 1] = child_idx.size();
        }
        if (child_idx.empty()) child_idx.push_back(0);
        const uint64_t n_ann = rnd() % 4;
        std::vector<uint64_t> ann_clade(n_ann + 1), ay(n_ann + 1, 0), aj(n_ann + 1, 0);
        std::string ytext, jtext;
        for (uint64_t a = 0; a < n_ann; ++a) {
            ann_clade[a] = rnd() % 50;
            ytext += "- clade: " + std::to_string(ann_clade[a]) + "\n"; ay[a + 1] = ytext.size();
            jtext += "{\"clade\":" + std::to_string(ann_clade[a]) + "}"; aj[a + 1] = jtext.size();
        }
        cls_record_tree rt{};
        rt.n_nodes = n_nodes; rt.node_id = node_id.data(); rt.parent_id = parent_id.data(); rt.node_kind = kind.data();
        rt.children_some = children_some.data(); rt.support = support.data(); rt.length = length.data(); rt.has_name = has_name.data();
        rt.name_off = name_off.data(); rt.names = names.data(); rt.child_off = child_off.data(); rt.child_idx = child_idx.data();
        rt.has_annotations = rnd() % 2; rt.n_annotations = n_ann; rt.ann_clade = ann_clade.data();
        rt.ann_yaml_off = ay.data(); rt.ann_yaml = ytext.data(); rt.ann_json_off = aj.data(); rt.ann_json = jtext.data();
        const uint64_t nq = rnd() % 5000;
        std::vector<uint8_t> status(nq + 1);
        std::vector<uint64_t> nid(nq + 1), hoff(nq + 1, 0);
        std::vector<int32_t> one(nq + 1), rest(nq + 1);
        std::vector<uint32_t> nroot(nq + 1);
        std::string headers;
        for (uint64_t q = 0; q < nq; ++q) {
            status[q] = (uint8_t)(rnd() % 11);
            nid[q] = node_id[rnd() % n_nodes];
            one[q] = (int32_t)rnd(); rest[q] = (int32_t)rnd(); nroot[q] = (uint32_t)rnd();
            headers += soup(rnd() % 20, 1);
            hoff[q + 1] = headers.size();
        }
        cls_result res{};
        res.status = status.data(); res.node_id = nid.data(); res.one = one.data(); res.rest = rest.data(); res.n_root_matched = nroot.data();
        for (uint32_t fmt = 0; fmt < 2; ++fmt) {
            char *o = nullptr, *e = nullptr;
            uint64_t no = 0, ne = 0;
            if (cls_records_render(&rt, nq, hoff.data(), headers.data(), &res, fmt, &o, &no, &e, &ne) != CLS_OK) { ++bad; continue; }
            if (!o || !e || o[no] != 0 || e[ne] != 0) ++bad;
            cls_text_free(o); cls_text_free(e);
        }
        cls_fasta_text_destroy(h);
    }
    printf("bad=%ld\n", bad);
    return bad ? 1 : 0;
}
