// Host-side model builder behind cls_model_build (include/classeq_b200.h): the k-mer -> node-set
// map of the reference's `map_kmers_to_tree` (core/src/use_cases/build_database/mod.rs:26-181)
// for one sequence per tip, each tip paired with its own sequence.  Offline, once per model;
// not part of the placement hot path (SURVEY.md section 8f, "next" row 4), but needed to manufacture
// the synthetic models of BASELINE.json's configs without going through multi-GB YAML.
#include <algorithm>
#include <atomic>
#include <cstring>
#include <memory>
#include <new>
#include <stdexcept>
#include <string>
#include <thread>
#include <unordered_map>
#include <vector>

#include "../../include/classeq_b200.h"
#include "built_model.hpp"
#include "host_pool.hpp"
#include "last_error.hpp"
#include "murmur3_host.hpp"

namespace {

struct Occ {
    uint64_t hash;
    uint64_t bucket;
    uint32_t tip;
};

inline uint64_t mix64(uint64_t x) { return cls::fmix64_h(x + 0x9e3779b97f4a7c15ULL); }

}  // namespace

static int build_host(const cls_model_view *tree, uint64_t n_tips, const uint64_t *tip_node,
                      const uint8_t *bases, const uint64_t *offsets, cls_built_model **out) {
    using cls::set_last_error;
    if (!tree || !out || (n_tips && (!tip_node || !offsets || !bases)))
        return set_last_error(CLS_ERR_INVALID_ARGUMENT, "NULL argument");
    *out = nullptr;
    const uint32_t k = tree->k_size, m = tree->m_size;
    if (k == 0) return set_last_error(CLS_ERR_UNSUPPORTED, "k_size == 0");
    const uint64_t n_nodes = tree->n_nodes;
    if (n_nodes == 0 || n_tips >= 0xFFFFFFFFull) return set_last_error(CLS_ERR_INVALID_ARGUMENT, "bad sizes");
    // parent links
    std::vector<int64_t> parent(n_nodes, -1);
    for (uint64_t p = 0; p < n_nodes; ++p)
        for (uint64_t j = tree->child_off[p]; j < tree->child_off[p + 1]; ++j) {
            if (tree->child_idx[j] >= n_nodes) return set_last_error(CLS_ERR_INVALID_ARGUMENT, "child index out of range");
            parent[tree->child_idx[j]] = (int64_t)p;
        }
    for (uint64_t t = 0; t < n_tips; ++t)
        if (tip_node[t] >= n_nodes) return set_last_error(CLS_ERR_INVALID_ARGUMENT, "tip node out of range");

    // ---- the inputs are not trusted: offsets must not decrease, sequences hold A/C/G/T only (either case: the
    //      reference upper-cases both strands, kmers_map.rs:410, and panics on anything else, :431-443) ----------
    for (uint64_t t = 0; t < n_tips; ++t)
        if (offsets[t] > offsets[t + 1]) return set_last_error(CLS_ERR_INVALID_ARGUMENT, "tip sequence offsets are not non-decreasing");
    {
        std::atomic<bool> bad{false};
        cls::parallel_for(n_tips, 64, [&](uint64_t a, uint64_t b) {
            for (uint64_t t = a; t < b; ++t)
                for (uint64_t i = offsets[t]; i < offsets[t + 1]; ++i) {
                    const uint8_t c = bases[i] & 0xDF;
                    if (!(c == 'A' || c == 'C' || c == 'G' || c == 'T')) { bad = true; return; }
                }
        });
        if (bad) return set_last_error(CLS_ERR_INVALID_ARGUMENT, "a tip sequence holds a character other than A, C, G, T");
    }

    // ---- all (hash, bucket, tip) occurrences, both strands (kmers_map.rs:375-398) ---------------
    std::vector<uint64_t> occ_off(n_tips + 1, 0);
    for (uint64_t t = 0; t < n_tips; ++t) {
        const uint64_t len = offsets[t + 1] - offsets[t];
        occ_off[t + 1] = occ_off[t] + (len >= k ? 2 * (len - k + 1) : 0);
    }
    std::vector<Occ> occ(occ_off[n_tips]);
    cls::parallel_for(n_tips, 1, [&](uint64_t t0, uint64_t t1) {   // the host pool carries exceptions back to this thread
        std::vector<uint8_t> fw, rc;
        for (uint64_t t = t0; t < t1; ++t) {
            const uint8_t *s = bases + offsets[t];
            const uint64_t len = offsets[t + 1] - offsets[t];
            if (len < k) continue;
            fw.resize(len); rc.resize(len);
            for (uint64_t i = 0; i < len; ++i) {
                const uint8_t c = s[i] & 0xDF;   // upper-case, both strands
                fw[i] = c;
                rc[len - 1 - i] = c == 'A' ? 'T' : c == 'T' ? 'A' : c == 'C' ? 'G' : 'C';
            }
            Occ *o = occ.data() + occ_off[t];
            const uint64_t W = len - k + 1;
            const uint32_t mm = std::min(m, k);
            for (int strand = 0; strand < 2; ++strand) {
                const uint8_t *d = strand ? rc.data() : fw.data();
                for (uint64_t i = 0; i < W; ++i) {
                    o->hash = cls::murmur3_x64_128_h1(d + i, k, 0);
                    // kmers_map.rs:131-137: key 0 when m_size == 0, else h1(first m chars)
                    o->bucket = m == 0 ? 0 : cls::murmur3_x64_128_h1(d + i, mm, 0);
                    o->tip = (uint32_t)t;
                    ++o;
                }
            }
        }
    });
    std::sort(occ.begin(), occ.end(), [](const Occ &a, const Occ &b) {
        if (a.hash != b.hash) return a.hash < b.hash;
        if (a.bucket != b.bucket) return a.bucket < b.bucket;
        return a.tip < b.tip;
    });

    // ---- group by (bucket, hash); de-duplicate tip lists; node set = union of root->tip paths ----
    std::unique_ptr<cls_built_model> guard(new cls_built_model());
    cls_built_model *bm = guard.get();
    bm->k_size = k; bm->m_size = m;
    bm->set_off.push_back(0);
    std::unordered_map<uint64_t, std::vector<uint64_t>> set_by_hash;  // tip-list hash -> set indices
    std::vector<std::vector<uint32_t>> set_tips;                       // kept only for equality checks
    std::vector<uint32_t> tips;
    std::vector<uint32_t> stamp(n_nodes, 0);
    uint32_t tag = 0;
    size_t i = 0;
    while (i < occ.size()) {
        size_t j = i;
        tips.clear();
        while (j < occ.size() && occ[j].hash == occ[i].hash && occ[j].bucket == occ[i].bucket) {
            if (tips.empty() || tips.back() != occ[j].tip) tips.push_back(occ[j].tip);
            ++j;
        }
        uint64_t h = 0x13198a2e03707344ULL;
        for (uint32_t t : tips) h = mix64(h ^ t);
        auto &cands = set_by_hash[h];
        uint64_t sid = ~0ull;
        for (uint64_t c : cands)
            if (set_tips[c] == tips) { sid = c; break; }
        if (sid == ~0ull) {
            sid = set_tips.size();
            set_tips.push_back(tips);
            cands.push_back(sid);
            if (++tag == 0) { std::fill(stamp.begin(), stamp.end(), 0); tag = 1; }
            for (uint32_t t : tips) {
                int64_t node = (int64_t)tip_node[t];
                while (node >= 0 && stamp[node] != tag) {
                    stamp[node] = tag;
                    bm->set_node_ids.push_back(tree->node_id[node]);
                    node = parent[node];
                }
            }
            bm->set_off.push_back(bm->set_node_ids.size());
        }
        bm->entry_bucket.push_back(occ[i].bucket);
        bm->entry_hash.push_back(occ[i].hash);
        bm->entry_set.push_back(sid);
        i = j;
    }
    *out = guard.release();
    return CLS_OK;
}

// Nothing is thrown across the ABI: host allocation failures become CLS_ERR_OUT_OF_MEMORY.
extern "C" int cls_model_build(const cls_model_view *tree, uint64_t n_tips, const uint64_t *tip_node,
                               const uint8_t *bases, const uint64_t *offsets, cls_built_model **out) {
    try {
        return build_host(tree, n_tips, tip_node, bases, offsets, out);
    } catch (const std::bad_alloc &) {
        if (out) *out = nullptr;
        return cls::set_last_error(CLS_ERR_OUT_OF_MEMORY, "host allocation failed while building the model");
    } catch (const std::exception &e) {
        if (out) *out = nullptr;
        return cls::set_last_error(CLS_ERR_INVALID_ARGUMENT, std::string("cls_model_build: ") + e.what());
    }
}

extern "C" int cls_built_model_view(const cls_built_model *bm, const cls_model_view *tree, cls_model_view *out) {
    if (!bm || !tree || !out) return cls::set_last_error(CLS_ERR_INVALID_ARGUMENT, "NULL argument");
    *out = *tree;
    out->k_size = bm->k_size;
    out->m_size = bm->m_size;
    out->n_entries = bm->entry_hash.size();
    out->entry_bucket = bm->entry_bucket.data();
    out->entry_hash = bm->entry_hash.data();
    out->entry_set = bm->entry_set.data();
    out->n_sets = bm->set_off.size() - 1;
    out->set_off = bm->set_off.data();
    out->set_node_ids = bm->set_node_ids.data();
    return CLS_OK;
}

extern "C" void cls_built_model_destroy(cls_built_model *bm) { delete bm; }
