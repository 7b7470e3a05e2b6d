// TEST INFRASTRUCTURE.  Memory-safety fuzz of the host-side model code under AddressSanitizer + UBSan: random - valid
// and malformed - cls_model_view inputs through build_host_index (classeq2_b200/csrc/index_build.cpp: what
// cls_index_create does before anything reaches the GPU) and random tip sets through cls_model_build (host_api.cpp).
// Malformed views must be REFUSED with an error code, never crash.  Built and run by tests/test_text_fuzz.py.
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <string>
#include <vector>

#include "../../include/classeq_b200.h"
#include "../../classeq2_b200/csrc/index_build.hpp"
#include "../../classeq2_b200/csrc/murmur3_host.hpp"

namespace cls {
int set_last_error(int code, const std::string &) { return code; }   // capi.cpp's, stubbed
}
extern "C" uint64_t cls_debug_host_murmur3_x64_128_h1(const uint8_t *d, uint64_t n, uint64_t s) { return cls::murmur3_x64_128_h1(d, n, s); }
extern "C" const char *cls_last_error(void) { return ""; }

static uint64_t rng_state = 0x9E3779B97F4A7C15ull;
static uint64_t rnd() { rng_state ^= rng_state << 13; rng_state ^= rng_state >> 7; rng_state ^= rng_state << 17; return rng_state; }

int main(int argc, char **argv) {
    const int rounds = argc > 1 ? atoi(argv[1]) : 400;
    long ok = 0, refused = 0;
    for (int r = 0; r < rounds; ++r) {
        const bool corrupt = r % 3 == 2;
        const uint64_t n = 1 + rnd() % 60;
        std::vector<uint64_t> node_id(n), child_off(n + 1, 0), child_idx;
        std::vector<uint8_t> kind(n);
        std::vector<std::vector<uint64_t>> kids(n);
        for (uint64_t i = 0; i < n; ++i) {
            node_id[i] = rnd() % 4 ? i * 3 + 1 : (rnd() >> (rnd() % 40));
            kind[i] = i == 0 ? CLS_KIND_ROOT : (rnd() % 2 ? CLS_KIND_LEAF : CLS_KIND_NODE);
            if (i) kids[rnd() % i].push_back(i);
        }
        for (uint64_t i = 0; i < n; ++i) {
            for (uint64_t c : kids[i]) child_idx.push_back(c);
            child_off[i + 1] = child_idx.size();
        }
        const uint64_t n_sets = 1 + rnd() % 30, n_entries = rnd() % 400;
        std::vector<uint64_t> set_off(n_sets + 1, 0), set_ids, eb(n_entries + 1), eh(n_entries + 1), es(n_entries + 1);
        for (uint64_t s = 0; s < n_sets; ++s) {
            const uint64_t m = rnd() % 8;
            for (uint64_t j = 0; j < m; ++j) set_ids.push_back(rnd() % 5 ? node_id[rnd() % n] : rnd() % 100);
            set_off[s + 1] = set_ids.size();
        }
        if (set_ids.empty()) set_ids.push_back(0);
        const uint32_t k = 1 + rnd() % 40, m_size = rnd() % 6;
        for (uint64_t e = 0; e < n_entries; ++e) {
            uint8_t pre[8];
            for (auto &c : pre) c = "ACGT"[rnd() & 3];
            eb[e] = m_size == 0 ? 0 : cls_debug_host_murmur3_x64_128_h1(pre, m_size < k ? m_size : k, 0);
            if (rnd() % 11 == 0) eb[e] = rnd();                          // unreachable bucket
            eh[e] = rnd();
            es[e] = rnd() % n_sets;
        }
        if (corrupt) {                                                     // one defect per round
            switch (rnd() % 8) {
                case 0: if (!child_idx.empty()) child_idx[rnd() % child_idx.size()] = n + rnd() % 5; break;
                case 1: if (!child_idx.empty()) child_idx[rnd() % child_idx.size()] = 0; break;
                case 2: if (child_idx.size() > 1) child_idx[0] = child_idx[1]; break;
                case 3: if (n > 1) node_id[1] = node_id[0]; break;
                case 4: if (n_entries) es[rnd() % n_entries] = n_sets + rnd() % 3; break;
                case 5: if (n_sets > 1) set_off[1] = set_off[n_sets] + 5; break;
                case 6: kind[rnd() % n] = 7; break;
                case 7: if (n_entries > 1) { eh[1] = eh[0]; eb[1] = eb[0]; } break;
            }
        }
        if (child_idx.empty()) child_idx.push_back(0);
        cls_model_view mv{};
        mv.k_size = k; mv.m_size = m_size; mv.flags = (uint32_t)(rnd() % 4);
        mv.n_nodes = n; mv.node_id = node_id.data(); mv.node_kind = kind.data(); mv.child_off = child_off.data(); mv.child_idx = child_idx.data();
        mv.n_entries = n_entries; mv.entry_bucket = eb.data(); mv.entry_hash = eh.data(); mv.entry_set = es.data();
        mv.n_sets = n_sets; mv.set_off = set_off.data(); mv.set_node_ids = set_ids.data();
        for (uint32_t shards : {1u, 3u}) {
            cls::HostIndex h;
            std::string err;
            const int rc = cls::build_host_index(&mv, h, err, shards - 1, shards);
            if (rc == CLS_OK) ++ok; else ++refused;
        }
        // ---- cls_model_build on a (valid) tree with random tips
        if (!corrupt) {
            const uint64_t n_tips = rnd() % 12;
            std::vector<uint64_t> tip_node(n_tips + 1), offsets(n_tips + 1, 0);
            std::string bases;
            for (uint64_t t = 0; t < n_tips; ++t) {
                tip_node[t] = rnd() % n;
                const uint64_t len = rnd() % 120;
                for (uint64_t j = 0; j < len; ++j) bases += "ACGTacgtN"[rnd() % 9];
                offsets[t + 1] = bases.size();
            }
            if (bases.empty()) bases = "A";
            cls_built_model *bm = nullptr;
            if (cls_model_build(&mv, n_tips, tip_node.data(), reinterpret_cast<const uint8_t *>(bases.data()), offsets.data(), &bm) == CLS_OK) {
                cls_model_view full{};
                cls_built_model_view(bm, &mv, &full);
                cls::HostIndex h;
                std::string err;
                if (cls::build_host_index(&full, h, err) == CLS_OK) ++ok; else ++refused;
                cls_built_model_destroy(bm);
            }
        }
    }
    printf("ok=%ld refused=%ld\n", ok, refused);
    return ok > 0 && refused > 0 ? 0 : 1;
}
